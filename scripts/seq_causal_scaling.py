"""Strong scaling of causal sequence sharding (zig-zag shards, gather strategy): one JSON line per workload.

    python -m torch.distributed.run --nproc-per-node N scripts/seq_causal_scaling.py [--steps 20] [--warmup 5]

Workloads: a Llama-3-8B layer at 128 k context (B1 Hq32 Hkv8 S131072 D128, causal) and BASELINE C3 (B1 H32 S8192
D128, causal).  Every rank builds the whole problem from one seed, times the unsharded one-GPU causal call
(``fp8_attn_func``) on its own GPU - the baseline of the efficiency - and then the sharded call on its zig-zag shard.
Per line: ms per step (CUDA events, after a warm-up, max over ranks), TFLOP/s (causal FLOPs halved, as
``oracle.attention_flops``), strong-scaling efficiency t1 / (N * tN), each rank's time inside the attention launches
(max over min: the zig-zag balance), cos and max-abs over row RMS of the sharded output against the unsharded one, GPU
name and power limit.  Inputs are far larger than L2.  Writes nothing but stdout.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import quantum_attn  # noqa: E402
from oracle import attention_flops  # noqa: E402
from quantumattention_b200 import parallel  # noqa: E402

WORKLOADS = {"llama3_8b_128k": (1, 32, 8, 131072, 128), "C3_llama": (1, 32, 32, 8192, 128)}


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def attend_ms(fn):
    """Time of one call inside its attention launches (from each head group's "wait" mark to its "attend" mark)."""
    parallel.trace_marks = []
    fn()
    torch.cuda.synchronize()
    marks, parallel.trace_marks = parallel.trace_marks, None
    return sum(a[1].elapsed_time(b[1]) for a, b in zip(marks, marks[1:]) if a[0] == "wait" and b[0] == "attend")


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in r.stdout.strip().split(",")]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", choices=sorted(WORKLOADS), action="append")
    ap.add_argument("--pv-mode", default=None, choices=["fp8", "fp8_hilo", "16bit"])
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    world, rank = dist.get_world_size(), dist.get_rank()
    pv = args.pv_mode or parallel.seq_pv_mode()
    name, power = gpu_info()
    for wl in args.workload or sorted(WORKLOADS):
        B, Hq, Hkv, S, D = WORKLOADS[wl]
        g = torch.Generator(device="cuda").manual_seed(0)
        q, k, v = (torch.randn(B, h, S, D, device="cuda", dtype=torch.bfloat16, generator=g) for h in (Hq, Hkv, Hkv))
        with quantum_attn.config.patch({"attention.pv_mode": pv}):
            one = lambda: quantum_attn.fp8_attn_func(q, k, v, is_causal=True)  # noqa: E731
            t1 = timed(one, max(5, args.steps // world), 2)
            whole = one()
        ref = parallel.zigzag_shard(whole, world, rank)
        del whole
        loc = [parallel.zigzag_shard(t, world, rank).contiguous() for t in (q, k, v)]
        del q, k, v
        call = lambda: parallel.ring_fp8_attention(*loc, is_causal=True, pv_mode=pv)  # noqa: E731
        dist.barrier()
        tn = timed(call, args.steps, args.warmup)
        out = call()
        a_ms = attend_ms(call) if world > 1 else tn
        # accuracy against the unsharded call, over the whole sequence
        o, r = out.float(), ref.float()
        row_rms = r.pow(2).mean(-1, keepdim=True).sqrt()
        acc = torch.stack([(o * r).sum(), (o * o).sum(), (r * r).sum()]).double()
        worst = ((o - r).abs() / row_rms).max().reshape(1)
        del o, r
        stats = torch.tensor([tn, a_ms, t1], device="cuda")
        every = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(every, stats)
        dist.all_reduce(acc)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        if rank == 0:
            every = torch.stack(every).cpu()
            t_n, t_1 = every[:, 0].max().item(), every[0, 2].item()
            att = every[:, 1]
            fl = attention_flops(B, Hq, S, S, D, True)
            print(json.dumps({
                "workload": wl, "shape": {"B": B, "Hq": Hq, "Hkv": Hkv, "S": S, "D": D, "causal": True}, "gpus": world,
                "pv_mode": pv, "strategy": "gather", "transport": parallel.default_seq_transport(),
                "peer_unavailable": parallel.last_transport_error(),
                "ms_per_step": round(t_n, 4), "tflops": round(fl / (t_n * 1e-3) / 1e12, 1),
                "one_gpu_ms": round(t_1, 4), "one_gpu_tflops": round(fl / (t_1 * 1e-3) / 1e12, 1),
                "strong_scaling_efficiency": round(t_1 / (world * t_n), 4),
                "attend_ms_per_rank": [round(x, 4) for x in att.tolist()],
                "attend_max_over_min": round((att.max() / att.min()).item(), 4),
                "cos_vs_unsharded": (acc[0] / (acc[1].sqrt() * acc[2].sqrt())).item(),
                "max_abs_over_row_rms_vs_unsharded": worst.item(),
                "steps": args.steps, "warmup": args.warmup, "gpu": name, "power_limit": power,
            }), flush=True)
        del loc, out, ref
        torch.cuda.empty_cache()
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
