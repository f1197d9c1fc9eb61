"""bench.py --dump-outputs on the GPU: the file holds what the last timed step returned, so that two builds of the
project can be compared output for output on the same seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
import quantum_attn

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    steps = 3
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C1", "--steps", str(steps), "--warmup", "1",
           "--pv-mode", "16bit", "--dump-outputs", str(tmp_path), "--no-comparators", "--no-cpu-baseline",
           "--no-other-modes", "--e2e-steps", "1"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    got = np.load(tmp_path / "out.npy")
    # bench.py rotates over input sets; on rank 0, set i is drawn from CPU seed i, and step i runs on set i
    B, H, S, D, causal = oracle.CONFIGS["C1"]
    g = torch.Generator(device="cpu").manual_seed(steps - 1)
    q, k, v = (torch.randn(B, H, S, D, generator=g, dtype=torch.float32).to(torch.bfloat16).cuda() for _ in range(3))
    with quantum_attn.config.patch({"attention.pv_mode": "16bit"}):
        want = quantum_attn.fp8_attn_func(q, k, v, is_causal=causal)
    assert got.dtype == np.float32 and np.array_equal(got, want.float().cpu().numpy())
