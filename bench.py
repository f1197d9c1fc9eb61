#!/usr/bin/env python
"""bench.py - FP8 attention forward throughput on B200 (the metric of BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload C2_flux|C3_llama|C1|C4_video] [--dump-outputs DIR]

One "step" = one call of the public entry point ``quantum_attn.fp8_attn_func(q, k, v)`` on 16-bit inputs that are
already resident in HBM: dynamic FP8 quantisation of Q/K/V plus the fused attention kernel - the same thing the
reference's own benchmark times (tests/test_interface.py:90-139).  FLOPs are the reference's formula, 4*B*H*Sq*Skv*D
(halved when causal, tests/test_interface.py:121-125).

Multi-GPU (torchrun, one rank per GPU): the path shards by batch x head with no collective, so every rank runs its
own batch element of the same workload (weak scaling); the time is the max over ranks.  The long-video workload
(C4_video) instead shards ONE sequence over the ranks (quantumattention_b200/parallel.py: one NCCL all-gather of the
e4m3 K/V under the local block's attention, or - QA_SEQ_STRATEGY=ring - neighbour send/recv; strong scaling).

``--impl reference`` times the reference's op definition (src/quantum_attn/ops.py:64-95: dequantise, aten SDPA) on the
box's host cores - the reference has no CPU kernel and its only GPU kernel is an sm_90a cubin that cannot load on
B200 (DESIGN.md).  Rank 0 only.
"""
import argparse
import json
import math
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (B, H, S, D, causal)  - BASELINE.json configs[0..2]
    "C1": (2, 8, 512, 64, True),
    "C2_flux": (1, 24, 4608, 128, False),
    "C3_llama": (1, 32, 8192, 128, True),
    # BASELINE.json configs[3]: Wan-720p token count; one GPU runs it whole, N GPUs shard the sequence (strong scaling; QA_SEQ_STRATEGY=gather|ring)
    "C4_video": (1, 24, 75600, 128, False),
}
METRIC = "fp8_attn_fwd_tflops"
UNIT = "TFLOP/s"
FP8_SPEC_TFLOPS = 4500.0


def flops_of(B, H, S, D, causal):
    f = 4 * B * H * S * S * D
    return f // 2 if causal else f


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.recording = threading.Event()  # samples are kept only while this is set (the timed region)
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if self.recording.is_set():
                    self.samples.append(mhz)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        return {
            "sm_mhz": statistics.median(self.samples) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
        }


def cpu_reference_leg(workload, budget_s=12.0, steps=None, warmup=1):
    """Time the reference's op definition on the host cores over a bounded sample of heads of the workload: ``steps``
    timed runs after ``warmup`` untimed ones, or, without ``steps``, as many runs (3 to 50) as fit in ``budget_s``."""
    import oracle

    B, H, S, D, causal = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    hs = 1 if S >= 8192 else min(H, 2)  # MATH materialises S x S per head: keep the sample bounded
    rows = S if S <= 16384 else 2048    # ... and for the video shape only a slab of query rows of that head
    q, k, v = oracle.make_qkv(1, hs, rows, S, D, seed=0)
    q8b, sq = oracle.quantize_fp8(q.float().numpy(), "head-wise")
    k8b, sk = oracle.quantize_fp8(k.float().numpy(), "head-wise")
    q8 = torch.from_numpy(q8b).view(torch.float8_e4m3fn)
    k8 = torch.from_numpy(k8b).view(torch.float8_e4m3fn)
    sq, sk, vf = torch.from_numpy(sq), torch.from_numpy(sk), v.float()
    for _ in range(warmup):
        oracle.cpu_reference_step(q8, k8, vf, sq, sk, is_causal=causal)
    times = []
    t_start = time.perf_counter()
    while (len(times) < steps if steps is not None else
           len(times) < 3 or (time.perf_counter() - t_start < budget_s and len(times) < 50)):
        t0 = time.perf_counter()
        oracle.cpu_reference_step(q8, k8, vf, sq, sk, is_causal=causal)
        times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    tflops = flops_of(1, hs, S, D, causal) * (rows / S) / t / 1e12
    return {
        "value": tflops, "unit": UNIT, "cores": cores, "kind": "port",
        "sample": f"{hs} of {B * H} heads of {workload} (S={S}, D={D}, causal={causal}"
                  + (f", {rows} of {S} query rows" if rows != S else "") + "), fp32 aten SDPA MATH on the "
                  f"dequantised inputs, median of {len(times)} runs; whole-workload time extrapolates linearly in heads",
        "seconds_per_sample": t,
    }


def fp8_gemm_peak(device):
    """Measured dense FP8 GEMM throughput (cuBLASLt through torch._scaled_mm), reported beside the spec figure."""
    try:
        n = 8192
        a = torch.randn(n, n, device=device).to(torch.float8_e4m3fn)
        b = torch.randn(n, n, device=device).to(torch.float8_e4m3fn).t()
        one = torch.tensor(1.0, device=device)
        for _ in range(3):
            torch._scaled_mm(a, b, scale_a=one, scale_b=one, out_dtype=torch.bfloat16)
        best = 1e9
        for _ in range(8):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._scaled_mm(a, b, scale_a=one, scale_b=one, out_dtype=torch.bfloat16)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2 * n**3 / (best * 1e-3) / 1e12
    except Exception:
        return None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line on the first
    collective): point file descriptor 1 at stderr for the duration of the run and keep the real stdout for the line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


DUMP_BYTES = 64 * 10**6


def dump_outputs(dirname, out):
    """Write ``out`` to dirname/out.npy as float32: whole when it fits in DUMP_BYTES, else the rows of its [B*H*S, D]
    view picked by torch.randperm under seed 0, in ascending order (the same rows for the same shape in every run)."""
    import numpy as np

    rows = out.reshape(-1, out.shape[-1])
    keep = (DUMP_BYTES - 4096) // (4 * rows.shape[1])  # (4096: room for the .npy header)
    if rows.shape[0] > keep:
        idx = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        out = rows[idx.to(rows.device)]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "out.npy"), out.float().cpu().numpy())


def accuracy_vs_sdpa(q, k, v, causal, out, heads=(0, -1), v_16bit=False):
    """BASELINE.json's "cos-sim vs ref": the output of the measured call against plain fp64 softmax(Q K^T) V (torch, on
    the GPU, outside every timed region) on the DEQUANTISED e4m3 inputs - the reference's op definition
    (src/quantum_attn/ops.py:64-95) carried to the FP8-V modes - for two heads of the workload.  north_star tolerance:
    cosine similarity >= 0.999, max-abs error <= 2e-2 of the output RMS (the latter is a bound for the hi+lo / 16-bit
    P modes; a single e4m3 P carries 2^-4 relative steps per probability)."""
    from quantumattention_b200 import _native

    (q8, k8, v8), (sq, sk, sv) = _native.quantize_fp8([q, k, v], _native.QA_SCALE_HEAD)
    D = q.shape[-1]
    cos, mx = [], []
    for h in heads:
        qd = q8[0, h].double() * sq[0, h].double()
        kd = k8[0, h].double() * sk[0, h].double()
        # (the 16-bit P/V mode is the reference's own op: V stays in its 16-bit dtype, only Q and K are dequantised)
        vd = v[0, h].double() if v_16bit else v8[0, h].double() * sv[0, h].double()
        sc = (qd @ kd.T) / math.sqrt(D)
        if causal:
            sc.masked_fill_(torch.ones_like(sc, dtype=torch.bool).triu_(1), float("-inf"))
        ref = torch.softmax(sc, dim=-1) @ vd
        got = out[0, h].double()
        cos.append(float((got * ref).sum() / (got.norm() * ref.norm())))
        # per-row RMS (tests/: oracle.compare's max_abs_over_row_rms): causal rows near the top are O(1), late rows small
        mx.append(float(((got - ref).abs() / ref.pow(2).mean(dim=-1, keepdim=True).sqrt()).max()))
        del sc
    return {"cos_sim": min(cos), "max_abs_over_row_rms": max(mx), "heads_checked": len(heads),
            "against": "fp64 softmax(QK^T)V on the dequantised e4m3 Q, K and " + ("16-bit V" if v_16bit else "e4m3 V") +
                       " (torch on the GPU, untimed)"}


def _slice_accuracy(out_rows, q8, k8, sq, sk, vd, rows, heads, D):
    """cos-sim / max-abs-over-row-RMS of `out_rows` [1,len(heads),len(rows),D] against fp64 softmax(QK^T/sqrt(D))V on the
    dequantised e4m3 Q / K and the value tensor `vd` (already dequantised or 16-bit), for the chosen heads and rows."""
    cos, mx = [], []
    for i, h in enumerate(heads):
        qd = q8[0, h][rows].double() * sq[0, h].double()
        kd = k8[0, h].double() * sk[0, h].double()
        ref = torch.softmax((qd @ kd.T) / math.sqrt(D), dim=-1) @ vd[i]
        got = out_rows[0, i].double()
        cos.append(float((got * ref).sum() / (got.norm() * ref.norm())))
        mx.append(float(((got - ref).abs() / ref.pow(2).mean(dim=-1, keepdim=True).sqrt()).max()))
    return {"cos_sim": min(cos), "max_abs_over_row_rms": max(mx)}


def seq_sharded_block(dev, rank, world, dist, steps, warmup):
    """BASELINE.json config 4 as ONE problem over all ranks (strong scaling): the long-video shape B1 H24 S75600 D128,
    sequence-sharded (quantumattention_b200/parallel.py).  Returns (on rank 0) the block that goes on the bench line:
    ms/step (max over ranks), TFLOP/s, strong-scaling efficiency against the same call on ONE GPU measured in this run,
    the transfer's bytes and achieved GB/s, a time split from CUDA events, and the accuracy of every P mode against the
    fp64 oracle on a slice (rank 0's first / middle / last 64 rows of two heads, all 75 600 keys)."""
    import quantum_attn
    from quantumattention_b200 import _native, parallel

    B, H, S, D, _ = WORKLOADS["C4_video"]
    if S % world:
        return {"skipped": f"S={S} does not split over {world} ranks"}
    S_loc = S // world
    pv_mode = parallel.seq_pv_mode()
    strategy, transport = parallel.default_seq_strategy(), parallel.default_seq_transport()

    def full_qkv():
        g = torch.Generator(device=dev).manual_seed(4321)  # same device type + seed on every rank: same sequence
        return [torch.randn((B, H, S, D), device=dev, dtype=torch.bfloat16, generator=g) for _ in range(3)]

    full = full_qkv()
    loc = [t[:, :, rank * S_loc:(rank + 1) * S_loc].contiguous() for t in full]
    del full

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(2, warmup // 4)):
        out = parallel.ring_fp8_attention(*loc)
    barrier()
    v_item = 2 if pv_mode == "16bit" else 1
    transport, comm = parallel.resolve_transport(transport, None, loc[0], loc[1], loc[2], v_item)  # what "auto" became
    transport_error = parallel.last_transport_error()
    n = max(5, min(steps, 30))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _native.launch_total
    barrier()
    e0.record()
    for _ in range(n):
        out = parallel.ring_fp8_attention(*loc)
    e1.record()
    barrier()
    launches = (_native.launch_total - l0) // n
    t = torch.tensor([e0.elapsed_time(e1) / n], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())

    # time split (separate untimed pass: the marks are CUDA events on the calling stream at the phase boundaries)
    split = None
    if strategy == "gather":
        # (calls issued back to back, the LAST one analysed: the host is then ahead of the GPU as in the timed loop)
        acc = {}
        reps = 4
        all_marks = []
        barrier()
        for _ in range(reps):
            parallel.trace_marks = []
            parallel.ring_fp8_attention(*loc)
            all_marks.append(parallel.trace_marks)
            parallel.trace_marks = None
        torch.cuda.synchronize()
        marks = all_marks[-1]
        prev_end = all_marks[-2][-1][1]
        acc["gap_after_previous_call"] = prev_end.elapsed_time(marks[0][1])
        waits = []
        for (_, a), (lb, b) in zip(marks, marks[1:]):
            acc[lb] = acc.get(lb, 0.0) + a.elapsed_time(b)
            if lb == "wait":
                waits.append(round(a.elapsed_time(b), 4))
        split = {("transfer_exposed" if k_ == "wait" else ("attention" if k_ == "attend" else k_)) + "_ms": v_
                 for k_, v_ in acc.items()}
        split["transfer_exposed_per_head_group_ms"] = waits
        split["note"] = ("one call of a back-to-back series, CUDA events on the compute stream: amax = local amax pass; scales = "
                         "all_reduce(MAX) of the head scales; quant_kv / quant_q = quantise with the global scales (K/V first: "
                         "they travel); transfer_exposed = time the compute stream waited for blocks; attention = the "
                         "per-head-group launches - or, gated_single_launch, the ONE launch over all heads whose CTAs "
                         "wait for their head group's blocks themselves (the first group's transfer is then inside it)")

    # the transfer alone, by the transport in use: every head group's blocks, nothing else running
    wire_bytes = (world - 1) * B * H * S_loc * D * (1 + v_item)  # received per rank per step
    chunks = parallel.head_chunks(B, H, S_loc)
    gather_ms = None
    try:
        if transport == "peer":
            main = torch.cuda.current_stream()
            for rep in range(4):
                barrier()
                if rep == 1:
                    e0.record()
                for evs in comm.pull(chunks):
                    for ev in evs:
                        main.wait_event(ev)
        else:
            k_loc = torch.empty((B, H, S_loc, D), dtype=torch.uint8, device=dev)
            v_loc = torch.empty((B, H, S_loc, D * v_item), dtype=torch.uint8, device=dev)
            k_all = torch.empty((B, H, S, D), dtype=torch.uint8, device=dev)
            v_all = torch.empty((B, H, S, D * v_item), dtype=torch.uint8, device=dev)
            for rep in range(4):
                barrier()
                if rep == 1:
                    e0.record()
                for lo, hi in chunks:
                    parallel._nccl_gather_heads([k_loc, v_loc], [k_all, v_all], lo, hi, None).wait()
            del k_loc, v_loc, k_all, v_all
        e1.record()
        barrier()
        tg = torch.tensor([e0.elapsed_time(e1) / 3], device=dev, dtype=torch.float64)
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        gather_ms = float(tg.item())
    except Exception as e:
        gather_ms = None
        transport_error = (transport_error or "") + " gather probe: " + repr(e)[:120]

    # accuracy of every P mode on a slice, and the same call on one GPU (rank 0 only; the others wait at the barrier)
    accuracy, one_gpu_ms = {}, None
    heads = [0, H - 1]
    rows = torch.cat([torch.arange(0, 64), torch.arange(S_loc // 2 - 32, S_loc // 2 + 32),
                      torch.arange(S_loc - 64, S_loc)]).to(dev)
    outs = {}
    for mode in ("16bit", "fp8_hilo", "fp8"):
        o = parallel.ring_fp8_attention(*loc, pv_mode=mode)
        outs[mode] = o[:, heads][:, :, rows].clone()
        del o
    barrier()
    if rank == 0:
        full = full_qkv()
        try:
            (q8, k8, v8), (sq, sk, sv) = _native.quantize_fp8([t[:, heads].contiguous() for t in full],
                                                              _native.QA_SCALE_HEAD)
            v16 = [full[2][0, h].double() for h in heads]
            vdq = [v8[0, i].double() * sv[0, i].double() for i in range(len(heads))]
            hs = list(range(len(heads)))
            for mode in ("16bit", "fp8_hilo", "fp8"):
                accuracy[mode] = _slice_accuracy(outs[mode], q8, k8, sq, sk, v16 if mode == "16bit" else vdq, rows,
                                                 hs, D)
            del q8, k8, v8, v16, vdq
        except Exception as e:
            accuracy = {"error": repr(e)[:200]}
        try:
            with quantum_attn.config.patch({"attention.pv_mode": pv_mode}):
                for i in range(3):
                    if i == 1:
                        e0.record()
                    quantum_attn.fp8_attn_func(*full)
                e1.record()
                torch.cuda.synchronize()
            one_gpu_ms = e0.elapsed_time(e1) / 2
        except Exception as e:
            one_gpu_ms = None
        del full
    barrier()
    if rank != 0:
        return None
    fl = flops_of(B, H, S, D, False)
    return {
        "workload": f"C4_video: ONE problem B={B} H={H} S={S} D={D} non-causal over {world} GPUs ({S_loc} tokens per rank)",
        "scaling": "strong", "n_gpus": world, "ms_per_step": ms, "steps": n, "value": fl / (ms * 1e-3) / 1e12, "unit": UNIT,
        "per_gpu_tflops": fl / (ms * 1e-3) / 1e12 / world, "pv_mode": pv_mode, "strategy": strategy,
        "transport": transport, "transport_error": transport_error, "head_groups": len(chunks),
        "gated_single_launch": bool(strategy == "gather" and transport == "peer" and parallel.seq_gated_launch(B, H, S_loc)),
        "gpu_launches_per_step": launches,
        "one_gpu_ms_same_run": one_gpu_ms,
        "strong_scaling_efficiency": (one_gpu_ms / (world * ms)) if one_gpu_ms else None,
        "wire": {"bytes_received_per_rank_per_step": wire_bytes,
                 "what": "e4m3 K + " + ("16-bit V" if v_item == 2 else "e4m3 V") + " blocks of the other ranks",
                 "gather_alone_ms": gather_ms,
                 "gather_alone_gbs": (wire_bytes / (gather_ms * 1e-3) / 1e9) if gather_ms else None,
                 "gather_alone_how": ("copy-engine pulls (qa_copy_2d from peer-mapped symmetric memory)" if transport == "peer"
                                      else "grouped NCCL all-gathers") + " of every head group back to back, nothing else "
                                     "running, max over ranks (measured reference on this pool: 770 GB/s peer copy per direction)"},
        "time_split": split,
        "accuracy": accuracy,
        "accuracy_against": "fp64 softmax(QK^T)V on the dequantised e4m3 Q, K and the mode's V (16-bit for '16bit', "
                            "dequantised e4m3 otherwise); rank 0's first / middle / last 64 rows of heads 0 and 23, all "
                            "75600 keys; bounds: cos >= 0.999, max-abs <= 2e-2 of the row RMS ('16bit', 'fp8_hilo')",
    }


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's threads to the CPUs of its GPU's NUMA node and prefer that node for new pages (the pinned
    staging buffers of the end-to-end leg), so host<->device copies do not cross the socket interconnect.  Best
    effort: reports what it could do.  (Round 1: all eight ranks ran on node 0 with buffers from one node and the
    end-to-end figure scaled 1.0 / 0.79 / 0.41 / 0.29 over 1 / 2 / 4 / 8 GPUs.)"""
    info = {"gpu_numa_node": None, "cpus_bound": None, "mempolicy": None}
    try:
        p = torch.cuda.get_device_properties(local_rank)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        info["gpu_numa_node"] = node
        if node < 0:
            return info
        cpus = set()
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if use:
            os.sched_setaffinity(0, use)
            info["cpus_bound"] = f"{len(use)} CPUs of node {node}"
        else:
            info["cpus_bound"] = f"none of node {node}'s CPUs is in this process's cpuset ({len(allowed)} allowed)"
        import ctypes
        libc = ctypes.CDLL("libc.so.6", use_errno=True)
        mask = ctypes.c_ulong(1 << node)
        rc = libc.syscall(238, 1, ctypes.byref(mask), 64)  # set_mempolicy(MPOL_PREFERRED, {node})
        info["mempolicy"] = f"preferred node {node}" if rc == 0 else f"set_mempolicy failed (errno {ctypes.get_errno()})"
    except Exception as e:
        info["error"] = repr(e)[:160]
    return info


def external_bars(sets, causal, fl, dev, workload=None):
    """On-box comparators (BASELINE.md section 6), rank 0, untimed extras: none of these is the reference, and none
    computes the reference's FP8 function - they are the bf16 / fp16 attention kernels of the stock libraries on the
    same shape, for scale.  Kernel-only, CUDA events, 10 launches after 3 warm-ups, rotating inputs."""
    import torch.nn.functional as F
    from torch.nn.attention import SDPBackend, sdpa_kernel

    res = {}

    def timeit(fn):
        for i in range(3):
            fn(*sets[i % len(sets)])
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(10):
            fn(*sets[i % len(sets)])
        b.record()
        torch.cuda.synchronize()
        return fl / (a.elapsed_time(b) / 10 * 1e-3) / 1e12

    for name, backend in (("torch_sdpa_cudnn_bf16", SDPBackend.CUDNN_ATTENTION), ("torch_sdpa_flash_bf16", SDPBackend.FLASH_ATTENTION)):
        try:
            def fn(q, k, v, _b=backend):
                with sdpa_kernel(_b):
                    return F.scaled_dot_product_attention(q, k, v, is_causal=causal)
            res[name] = timeit(fn)
        except Exception as e:
            res[name] = "unavailable: " + repr(e)[:100]
    try:
        from flash_attn import flash_attn_func

        bshd = [tuple(t.transpose(1, 2).contiguous() for t in s_) for s_ in sets[:2]]

        def fa(q, k, v):
            return flash_attn_func(q, k, v, causal=causal)
        for i in range(3):
            fa(*bshd[i % 2])
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(10):
            fa(*bshd[i % 2])
        b.record()
        torch.cuda.synchronize()
        res["flash_attn_2_bf16"] = fl / (a.elapsed_time(b) / 10 * 1e-3) / 1e12
        del bshd
    except Exception as e:
        res["flash_attn_2_bf16"] = "unavailable: " + repr(e)[:100]
    try:
        import flashinfer

        bshd = [tuple(t[0].transpose(0, 1).contiguous() for t in s_) for s_ in sets[:2]]  # [S, H, D]

        def fi(q, k, v):
            return flashinfer.single_prefill_with_kv_cache(q, k, v, causal=causal)
        for i in range(3):
            fi(*bshd[i % 2])
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(10):
            fi(*bshd[i % 2])
        b.record()
        torch.cuda.synchronize()
        res["flashinfer_single_prefill_bf16"] = fl / (a.elapsed_time(b) / 10 * 1e-3) / 1e12
        del bshd
    except Exception as e:
        res["flashinfer_single_prefill_bf16"] = "unavailable: " + repr(e)[:100]
    # NVIDIA's CuTe-DSL Blackwell FMHA example (shipped inside the flashinfer wheel), FP8 and fp16 inputs, in a process of
    # its own (it JIT-compiles; ~10 s per variant) - a comparator, not the reference and not product code
    if workload in ("C2_flux", "C3_llama"):
        try:
            import subprocess
            out_ = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "cutedsl_fmha_bar.py"), workload],
                                  capture_output=True, text=True, timeout=180).stdout
            line_ = [ln for ln in out_.splitlines() if ln.startswith("CUTEDSL_JSON ")][-1]
            for k_, v_ in json.loads(line_[len("CUTEDSL_JSON "):]).items():
                res["cutedsl_fmha_" + k_.split("_", 2)[-1].lower()] = v_.get("tflops", "unavailable: " + str(v_.get("error")))
        except Exception as e:
            res["cutedsl_fmha"] = "unavailable: " + repr(e)[:100]
    res["unit"] = UNIT
    res["note"] = ("stock attention kernels on the same shape and FLOP count, kernel only: bf16 cuDNN / flash / flash_attn / "
                   "flashinfer, and NVIDIA's CuTe-DSL Blackwell FMHA example with Float8E4M3FN and Float16 inputs (its own "
                   "benchmark loop); none of them computes the reference's mixed FP8 / 16-bit function")
    return res


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 1000, or 30 for sequences over 16k tokens); the reference arm times this "
                         "many runs of its sample")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (rank 0) to DIR/out.npy as float32; "
                         "an output over 64 MB is cut to its rows [B*H*S, D] of a seed-0 sample, in order")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2_flux", choices=sorted(WORKLOADS))
    ap.add_argument("--event-every", type=int, default=None,
                    help="bracket the attention kernel with CUDA events on every N-th timed step (the two event records "
                         "cost about 6 us of GPU time per bracketed step on C2; 1 = every step; default 8, or 4 for "
                         "runs of fewer than 100 steps so that a short run still has several samples)")
    ap.add_argument("--no-seq-sharded", action="store_true",
                    help="N > 1: skip the C4 strong-scaling block (one sequence sharded over all ranks)")
    ap.add_argument("--no-comparators", action="store_true", help="skip the stock-library attention kernels")
    ap.add_argument("--pv-mode", default=None, choices=["fp8", "fp8_hilo", "16bit"])
    ap.add_argument("--e2e-steps", type=int, default=40)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-modes", action="store_true", help="skip the kernel-only numbers of the other P modes")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    B, H, S, D, causal = WORKLOADS[args.workload]
    ring = args.workload == "C4_video" and world > 1
    if args.steps is None:
        args.steps = 1000 if S <= 16384 else 30
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.event_every is None:
        args.event_every = 8 if args.steps >= 100 else 4
    if S > 16384:
        args.e2e_steps = min(args.e2e_steps, 10)
    # (everything in `config` is a function of the command line and the environment alone, so the reference arm of
    # the same command prints the same dict)
    pv_mode = args.pv_mode or os.getenv("QUANTUM_ATTN_PV_MODE", "16bit")
    bytes_per_set = 3 * B * H * (S // world if ring else S) * D * 2
    n_sets = max(2, math.ceil(300e6 / bytes_per_set))
    config = {
        "workload": f"{args.workload}: B={B} (per GPU) H={H} S={S} D={D} causal={causal}, head-wise FP8 scales",
        "per_gpu_batch": B, "heads": H, "seq_len": S, "head_dim": D, "causal": causal,
        "parallelism": f"batch x head sharding over {world} GPU(s), no collective",
        "l2_policy": f"rotating {n_sets} input sets ({n_sets * bytes_per_set / 1e6:.0f} MB > 126 MB L2)",
        "kernel_timing": (f"CUDA events around the attention launch of every {args.event_every}-th timed step, on its "
                          "stream (roofline.achieved is their mean)"),
        "pv_mode": pv_mode,
    }
    if ring:
        if S % world:
            raise SystemExit(f"bench.py: S={S} does not split over {world} ranks")
        config["workload"] = (f"{args.workload}: ONE problem B={B} H={H} S={S} D={D} causal={causal} over {world} GPUs, "
                              f"{S // world} tokens per rank, head-wise FP8 scales (global via all_reduce MAX)")
        from quantumattention_b200.parallel import default_seq_strategy, default_seq_transport
        config["parallelism"] = (
            f"sequence sharding over {world} GPUs: e4m3 K (+ V) blocks by NCCL send/recv ring, (O, LSE) merge per block"
            if default_seq_strategy() == "ring" else
            f"sequence sharding over {world} GPUs: every rank's K / V blocks gathered per head group into the kernel's "
            f"layout ({default_seq_transport()} transport), one launch per head group over all keys, no merge")
        config["seq_strategy"] = default_seq_strategy()
        config["seq_transport"] = default_seq_transport()

    # ------------------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        W = max(args.warmup, 0)
        leg = cpu_reference_leg(args.workload, steps=args.steps, warmup=W)
        line = {
            "impl": "reference", "metric": METRIC, "value": leg["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": W, "ms_per_step": leg["seconds_per_sample"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": leg["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line), file=out, flush=True)
        return

    # ------------------------------------------------------------------------------ our arm (B200)
    import quantum_attn
    from quantumattention_b200 import _native

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sm_100a path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    quantum_attn.config.attention.pv_mode = pv_mode
    _native.load(build_if_missing=False)
    host_binding = bind_to_gpu_numa_node(local_rank)

    # rotating input sets so the working set (> 126 MB L2) is not L2-resident between steps

    def make_qkv(seed):  # SURVEY 8(d): CPU-generated randn so every run (and the CPU arm) sees the same bits
        g = torch.Generator(device="cpu").manual_seed(seed)
        return tuple(torch.randn(B, H, S, D, generator=g, dtype=torch.float32).to(torch.bfloat16) for _ in range(3))

    S_loc = S // world if ring else S
    sets = []
    for i in range(n_sets):
        if ring:  # every rank generates the same sequence and keeps its slice
            q, k, v = (t[:, :, rank * S_loc:(rank + 1) * S_loc].contiguous() for t in make_qkv(i))
        else:
            q, k, v = make_qkv(1000 * rank + i)
        sets.append((q.to(dev), k.to(dev), v.to(dev)))

    from quantumattention_b200 import parallel

    def attn_call(q, k, v):
        if ring:
            return parallel.ring_fp8_attention(q, k, v)
        return quantum_attn.fp8_attn_func(q, k, v, is_causal=causal)

    def step(i):
        return attn_call(*sets[i % n_sets])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # the NVML sampler thread is started BEFORE the warm-up (NVML initialisation and its first queries take driver
    # locks the launch path also wants: inside a 4 ms timed region that showed up as 10-20 us per step); it keeps
    # samples only while `recording` is set
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(max(args.warmup, 3)):
        step(i)
    barrier()

    sampler.recording.set()
    _native.attn_events = []
    launches0 = _native.launch_total
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    ev_list = _native.attn_events
    for i in range(args.steps):
        # the attention launch of every `--event-every`-th step is bracketed by CUDA events (roofline.achieved)
        _native.attn_events = ev_list if i % args.event_every == 0 else None
        last_out = step(i)
        if i + 1 < args.steps:
            del last_out  # (freed as it returns, so the allocator serves every step from the same cached blocks)
    _native.attn_events = ev_list
    e1.record()
    launches = _native.launch_total - launches0
    # a short timed region (the driver's 20 steps are 4 ms) holds one NVML sample at best: keep the same steps running,
    # untimed, until the sampler has seen half a second of this load
    t_wall = time.perf_counter()
    _native.attn_events = None
    extra_steps = 0
    while not ring and time.perf_counter() - t_wall < 0.5 and args.steps * (S / 4608.0) ** 2 < 400:
        step(extra_steps)
        extra_steps += 1
        if extra_steps % 64 == 0:
            torch.cuda.synchronize()
    _native.attn_events = ev_list
    barrier()
    total_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    clocks["sampled_over"] = ("the timed region" if extra_steps == 0 else
                              f"the timed region and {extra_steps} identical untimed steps right after it")
    events, _native.attn_events = _native.attn_events, None
    attn_ms = statistics.mean(a.elapsed_time(b) for a, b in events)
    if rank == 0 and args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, last_out)
    del last_out

    if dist is not None:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    fl = flops_of(B, H, S, D, causal)
    job_fl = fl if ring else world * fl  # the ring splits ONE problem; head/batch sharding replicates the workload
    value = job_fl / (ms_per_step * 1e-3) / 1e12

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timed region.
    # Every step copies its own q, k, v from pinned host memory and reads its own output back.  The three legs run on
    # three streams with double-buffered device tensors, so step i+1's upload and step i-1's download overlap step
    # i's kernels (PCIe is full duplex); the region is timed with events from before the first upload to after the
    # last download.
    hq, hk, hv = (t.cpu().pin_memory() for t in sets[0])
    houts = [torch.empty_like(hq).pin_memory() for _ in range(2)]
    dbuf = [tuple(torch.empty_like(t) for t in sets[0]) for _ in range(2)]
    s_main = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def e2e_run(n):
        up = [None, None]        # upload-finished events per buffer
        done = [None, None]      # compute-finished events per buffer (the buffer may be overwritten after it)
        down = [None, None]      # download-finished events per host output buffer
        outs = [None, None]
        for i in range(n):
            b_ = i & 1
            with torch.cuda.stream(s_in):
                if done[b_] is not None:
                    s_in.wait_event(done[b_])
                for d, h_ in zip(dbuf[b_], (hq, hk, hv)):
                    d.copy_(h_, non_blocking=True)
                up[b_] = torch.cuda.Event()
                up[b_].record(s_in)
            s_main.wait_event(up[b_])
            if down[b_] is not None:
                s_main.wait_event(down[b_])  # outs[b_] of two steps ago has been read back
            outs[b_] = attn_call(*dbuf[b_])
            done[b_] = torch.cuda.Event()
            done[b_].record(s_main)
            with torch.cuda.stream(s_out):
                s_out.wait_event(done[b_])
                houts[b_].copy_(outs[b_], non_blocking=True)
                down[b_] = torch.cuda.Event()
                down[b_].record(s_out)
        for ev in down:
            if ev is not None:
                s_main.wait_event(ev)

    e2e_run(3)
    barrier()
    s_in.wait_stream(s_main)
    e0.record()
    s_in.wait_event(e0)
    e2e_run(args.e2e_steps)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = job_fl / (e2e_ms / args.e2e_steps * 1e-3) / 1e12
    # host link per rank, all ranks copying at once (what bounds the end-to-end figure): one direction at a time
    link = {}
    for name, dst_, src_, strm in (("h2d_gbs", dbuf[0][0], hq, s_in), ("d2h_gbs", houts[0], dbuf[0][0], s_out)):
        barrier()
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(strm):
            a_.record(strm)
            for _ in range(8):
                dst_.copy_(src_, non_blocking=True)
            b_.record(strm)
        barrier()
        link[name] = 8 * hq.numel() * hq.element_size() / (a_.elapsed_time(b_) * 1e-3) / 1e9
    if dist is not None:
        lt = torch.tensor([link["h2d_gbs"], link["d2h_gbs"]], device=dev, dtype=torch.float64)
        allv = [torch.empty_like(lt) for _ in range(world)]
        dist.all_gather(allv, lt)
        link = {"h2d_gbs_per_rank": [round(float(x[0]), 1) for x in allv],
                "d2h_gbs_per_rank": [round(float(x[1]), 1) for x in allv]}
    link["how"] = "8 back-to-back copies of one pinned [B,H,S,D] bf16 tensor per direction, every rank at the same time"
    bindings = [host_binding]
    if dist is not None:
        bindings = [None] * world
        dist.all_gather_object(bindings, host_binding)

    # ---- the quantiser alone (HBM-bound leg of the step): Q, K, V of one input set per launch, rotating sets
    quant_ms = None
    if rank == 0:
        qmode = _native.QA_SCALE_HEAD
        nq = 2 if pv_mode == "16bit" else 3  # what the step's own quantiser launch covers in this mode
        for i in range(3):
            _native.quantize_fp8(list(sets[i % n_sets])[:nq], qmode)
        torch.cuda.synchronize()
        # mean launch duration over back-to-back launches on rotating sets, replayed from a CUDA graph so that no host
        # time sits between them (a Python call of the binding costs about as much as the kernel runs; a CUDA-event
        # pair per launch adds ~6 us of event-record time to a ~25 us kernel)
        n_q = 4 * n_sets
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            _native.quantize_fp8(list(sets[0])[:nq], qmode)
        torch.cuda.current_stream().wait_stream(side)
        qgraph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(qgraph):
            for i in range(n_q):
                _native.quantize_fp8(list(sets[i % n_sets])[:nq], qmode)
        qgraph.replay()
        torch.cuda.synchronize()
        qa_, qb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        qa_.record()
        for _ in range(5):
            qgraph.replay()
        qb_.record()
        torch.cuda.synchronize()
        quant_ms = qa_.elapsed_time(qb_) / (5 * n_q)
        del qgraph
        # host-side cost of one step (python + ctypes + allocator), GPU not waited for (not in ring mode: a step
        # there holds collectives and every rank would have to take part)
        host_us = None
        if not ring:
            host_us = 1e9
            for _ in range(4):  # best of four bursts of 30 calls (a burst can catch a collection or an allocator refill)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for i in range(30):
                    step(i)
                host_us = min(host_us, (time.perf_counter() - t0) / 30 * 1e6)
            torch.cuda.synchronize()

    # ---- the other two P modes, kernel only (context for the headline mode; 20 launches each)
    other_modes, other_steps = {}, {}
    if rank == 0 and not args.no_other_modes and not ring:
        for mode in ("fp8", "fp8_hilo", "16bit"):
            if mode == pv_mode:
                continue
            with quantum_attn.config.patch({"attention.pv_mode": mode}):
                for i in range(3):
                    step(i)
                _native.attn_events = []
                for i in range(20):
                    step(i)
                torch.cuda.synchronize()
                ev, _native.attn_events = _native.attn_events, None
                other_modes[mode] = fl / (statistics.mean(a.elapsed_time(b) for a, b in ev) * 1e-3) / 1e12
                # and the whole step (quantise + attention, no per-launch events), 100 back-to-back steps
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                for i in range(100):
                    step(i)
                s1.record()
                torch.cuda.synchronize()
                other_steps[mode] = fl / (s0.elapsed_time(s1) / 100 * 1e-3) / 1e12
        # the 16-bit entry point (`attn_func`: bf16 Q / K / V, kind::f16 MMAs, no quantiser), same shape and FLOP count
        for i in range(3):
            quantum_attn.attn_func(*sets[i % n_sets], is_causal=causal)
        _native.attn_events = []
        for i in range(20):
            quantum_attn.attn_func(*sets[i % n_sets], is_causal=causal)
        torch.cuda.synchronize()
        ev, _native.attn_events = _native.attn_events, None
        other_modes["attn_func_bf16"] = fl / (statistics.mean(a.elapsed_time(b) for a, b in ev) * 1e-3) / 1e12

    comparators = None
    if rank == 0 and world == 1 and not args.no_comparators and S <= 16384:
        try:
            comparators = external_bars(sets, causal, fl, dev, args.workload)
        except Exception as e:
            comparators = {"error": repr(e)[:200]}

    accuracy = None
    if rank == 0 and not ring:
        try:
            accuracy = accuracy_vs_sdpa(*sets[0], causal, attn_call(*sets[0]), v_16bit=(pv_mode == "16bit"))
            accuracy["pv_mode"] = pv_mode
            if pv_mode != "fp8_hilo":  # the mode that is built to meet the 2e-2 max-abs bound, for comparison
                with quantum_attn.config.patch({"attention.pv_mode": "fp8_hilo"}):
                    hl = accuracy_vs_sdpa(*sets[0], causal, attn_call(*sets[0]))
                accuracy["fp8_hilo"] = {k_: hl[k_] for k_ in ("cos_sim", "max_abs_over_row_rms")}
        except Exception as e:  # a reporting extra: never lose the bench line to it
            accuracy = {"error": repr(e)[:200]}

    seq_block = None
    if world > 1 and not args.no_seq_sharded:
        del sets, dbuf, hq, hk, hv, houts
        torch.cuda.empty_cache()
        try:
            seq_block = seq_sharded_block(dev, rank, world, dist, args.steps, args.warmup)
        except Exception as e:  # never lose the main line to the extra block
            seq_block = {"error": repr(e)[:300]}
        sets = None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    fp8_meas = fp8_gemm_peak(dev)
    if ring:
        # launches per step: one per head group over all keys (gather) or one per key block (ring); every launch of a
        # step does the same share of the rank's FLOPs (fl / world)
        from quantumattention_b200.parallel import default_seq_strategy, head_chunks
        n_l = len(head_chunks(B, H, S_loc)) if default_seq_strategy() == "gather" else world
        launch_fl = fl // world // n_l
    else:
        launch_fl = fl
    achieved = launch_fl / (attn_ms * 1e-3) / 1e12
    # The driver measures bf16 only; kind::f8f6f4 runs at exactly twice the bf16 rate on the same datapath, so the
    # FP8 denominator is 2 x the MEASURED bf16 GEMM burst figure.  Spec and measured-FP8-GEMM fractions sit beside it.
    peak = 2.0 * peaks["bf16_tflops"]
    peak_note = "2 x bf16_tflops"
    if pv_mode == "16bit":
        # half of the launch's FLOPs (Q K^T) run as kind::f8f6f4, half (P V) as kind::f16 at the bf16 rate: the tensor
        # roofline of that mix is the harmonic combination 1 / (0.5 / (2 P16) + 0.5 / P16) = 4/3 x the bf16 figure
        peak = peaks["bf16_tflops"] * 4.0 / 3.0
        peak_note = "4/3 x bf16_tflops (Q K^T at the FP8 rate = 2 x bf16, P V at the bf16 rate, equal FLOPs)"
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(args.workload, {}).get(pv_mode)
        except Exception:
            traffic = None
    roofline = {
        "kernel": "attn_fwd_kernel", "bound": "tensor", "achieved": achieved, "peak": peak, "unit": UNIT,
        "frac": achieved / peak, "traffic": traffic,
        "traffic_source": "profiles/roofline_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of this kernel "
                          "from an `ncu --set full` capture of this workload and mode (static, not measured in this run)",
        "kernel_samples": len(events),
        "peak_source": f"{peak_note} ({peaks['source']} MEASURED_PEAKS.json burst {peaks['bf16_tflops']}); "
                       "the file holds no FP8 figure",
        "frac_of_fp8_spec_4500": achieved / FP8_SPEC_TFLOPS,
        "fp8_gemm_tflops_measured_here": fp8_meas,
        "frac_of_measured_fp8_gemm": (achieved / fp8_meas) if fp8_meas else None,
        "attn_kernel_ms": attn_ms, "flops_per_launch": launch_fl,
        "exp_bound_tflops_at_max_clock": 148 * 16 * 1.965e9 * 4 * D / 1e12,
    }
    n_quant = 2 if pv_mode == "16bit" else 3  # V stays 16-bit in the reference's mode: only Q and K are quantised
    quant_bytes = n_quant * B * H * S_loc * D * 3 + n_quant * B * H * 4  # 2 B in + 1 B out per element, + scales (SURVEY 8d)
    quantiser = {
        "kernel": "quant_head_ring_kernel", "bound": "hbm", "ms": quant_ms,
        "how": "mean launch duration over back-to-back launches on rotating input sets (> L2), replayed from a CUDA graph "
               "(no host time between launches; each launch clears its scratch workspace), one CUDA-event pair round the lot",
        "achieved": quant_bytes / (quant_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
        "frac": quant_bytes / (quant_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes": quant_bytes,
        "traffic": None,
    }
    try:
        tq = json.load(open(tpath)).get("quantiser", {})
        quantiser["traffic"] = tq.get("quant_head_ring_kernel")
    except Exception:
        pass
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if ring else "weak", "vs_baseline": None,
        "dtype": "fp8_e4m3" if pv_mode != "16bit" else "fp8_e4m3(QK^T)+bf16(PV), the reference's", "data": "synthetic",
        "config": config, "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 3 * B * H * S_loc * D * 2,
                "d2h_bytes_per_step": B * H * S_loc * D * 2, "ms_per_step": e2e_ms / args.e2e_steps},
        "roofline": roofline,
        "quantiser": quantiser,
        "host_us_per_step": host_us,
        "per_gpu_tflops": value / world,
        "frac_of_fp8_spec": value / world / FP8_SPEC_TFLOPS,
        "other_pv_modes_kernel_tflops": other_modes,
        "other_pv_modes_step_tflops": other_steps,
        "accuracy": accuracy,
        "comparators": comparators,
        "host_link": link,
        "host_binding": bindings,
    }
    if seq_block is not None:
        line["seq_sharded"] = seq_block
    if world == 1 and not args.no_cpu_baseline:
        leg = cpu_reference_leg(args.workload)
        line["cpu_baseline"] = {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), file=out, flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
