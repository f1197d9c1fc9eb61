"""Developer tool: head-wise quantiser, mean launch duration over back-to-back launches replayed from a CUDA graph
(no host time between launches).  Shapes: Q and K of C2 / C3, Q K V of C4 and of the S >= 32 k sweep entries."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from quantumattention_b200 import _native
dev = torch.device("cuda:0")
for name, (H, S, D, n) in {"C2": (24, 4608, 128, 2), "C3": (32, 8192, 128, 2), "C4": (24, 75600, 128, 3), "C4qk": (24, 75600, 128, 2),
                            "s32k": (8, 32768, 128, 3), "s128k": (2, 131072, 128, 3), "d256s64k": (4, 65536, 256, 3)}.items():
    nsets = 3 if S * H < 1e6 else 2
    sets = [[torch.randn((1, H, S, D), device=dev, dtype=torch.bfloat16) for _ in range(n)] for _ in range(nsets)]
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        _native.quantize_fp8(sets[0], _native.QA_SCALE_HEAD)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    reps = 6
    with torch.cuda.graph(g):
        for i in range(reps):
            _native.quantize_fp8(sets[i % nsets], _native.QA_SCALE_HEAD)
    nl = _native.last_launch_count()
    g.replay(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(4):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / (4 * reps)
    by = n * H * S * D * 3
    print(f"{name}: {ms * 1e3:7.1f} us  {by / ms / 1e6:6.0f} GB/s  launches/call {nl}", flush=True)
    del sets, g
