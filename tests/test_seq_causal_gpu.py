"""Causal and GQA sequence sharding against the unsharded one-GPU call: every rank's launches on one GPU, and the
whole path on two GPUs.

Causal: zig-zag shards (``parallel.zigzag_shard``), K / V gathered in global token order, each head group attended in
two bottom-right launches.  The chunk (640 rows) is a multiple of the kernel's 128-row query tile, so every query tile
of a sharded launch covers the rows of one tile of the unsharded launch, with the same keys, the same 64-key steps and
the same quantised bytes (the head scales are made global by one MAX all-reduce): the result is bit for bit the
unsharded ``fp8_attn_func(..., is_causal=True)``.  Non-causal GQA through the gather strategy likewise (only the Hkv
heads of K / V travel).  Both transports, three repeated calls (the peer transport alternates its two send slots),
every P mode."""
import math
import os
import socket

import pytest
import torch

import oracle
import quantum_attn
from quantumattention_b200 import _native, parallel

pytestmark = pytest.mark.gpu

B, HQ, HKV, C, D = 1, 8, 2, 640, 128


@pytest.mark.parametrize("world", [2, 4, 8])
def test_zigzag_launches_of_every_rank_equal_the_unsharded_launch(world):
    """What each rank of a causal gather launches, minus the wire, on one GPU: the two bottom-right launches of rank r
    (chunk r over the first (r + 1) c keys, chunk 2N-1-r over the first (2N - r) c keys, on views of K / V in global
    token order and of the zig-zag Q) give, bit for bit, the rows of the unsharded causal launch - GQA, every P mode."""
    c = C
    S = 2 * world * c
    q, k, v = (t.cuda() for t in _inputs(world))
    (q8,), (sq,) = _native.quantize_fp8([q], _native.QA_SCALE_HEAD)
    (k8, v8), (sk, sv) = _native.quantize_fp8([k, v], _native.QA_SCALE_HEAD)
    for mode, p_mode in (("16bit", _native.QA_P_16BIT), ("fp8", _native.QA_P_E4M3), ("fp8_hilo", _native.QA_P_E4M3_HILO)):
        vin, svin = (v, None) if mode == "16bit" else (v8, sv)
        kw = dict(scale_mode=_native.QA_SCALE_HEAD, sm_scale=1 / math.sqrt(D), p_mode=p_mode, out_dtype=torch.bfloat16)
        whole = _native.fp8_attn_fwd(q8, k8, vin, sq, sk, svin, is_causal=True, **kw)
        for r in range(world):
            q_loc = parallel.zigzag_shard(q8.view(torch.uint8), world, r).view(torch.float8_e4m3fn)
            for rows, first, n_keys in ((slice(0, c), r * c, (r + 1) * c), (slice(c, 2 * c), (2 * world - 1 - r) * c,
                                                                            (2 * world - r) * c)):
                o = _native.fp8_attn_fwd(q_loc[:, :, rows], k8[:, :, :n_keys], vin[:, :, :n_keys], sq, sk, svin,
                                         is_causal=_native.QA_CAUSAL_BOTTOM_RIGHT, **kw)
                assert torch.equal(o, whole[:, :, first:first + c]), (world, r, first, mode)
        assert S == whole.shape[2]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _inputs(world):
    S = 2 * world * C
    g = torch.Generator().manual_seed(21)
    q, k, v = (torch.randn(B, h, S, D, generator=g).to(torch.bfloat16) for h in (HQ, HKV, HKV))
    return q, k * torch.linspace(0.5, 2.0, S).view(1, 1, -1, 1).to(k.dtype), v


def _worker(rank, world, port, tmp):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        q, k, v = (t.cuda() for t in _inputs(world))
        S_local = 2 * C
        res, peer_error = {}, None
        for pv in ("16bit", "fp8", "fp8_hilo"):
            with quantum_attn.config.patch({"attention.pv_mode": pv}):
                whole_c = parallel.zigzag_shard(quantum_attn.fp8_attn_func(q, k, v, is_causal=True), world, rank)
                whole_n = quantum_attn.fp8_attn_func(q, k, v)[:, :, rank * S_local:(rank + 1) * S_local]
            loc_c = [parallel.zigzag_shard(t, world, rank).contiguous() for t in (q, k, v)]
            loc_n = [t[:, :, rank * S_local:(rank + 1) * S_local].contiguous() for t in (q, k, v)]
            for causal, transport, gated in ((True, "nccl", "0"), (True, "peer", "0"), (False, "nccl", "0"),
                                             (False, "peer", "1"), (False, "peer", "0")):
                if transport == "peer" and peer_error is not None:
                    continue
                os.environ["QA_SEQ_GATED"] = gated  # (the causal path never takes the gated launch)
                try:
                    for rep in range(3):
                        out = parallel.ring_fp8_attention(*(loc_c if causal else loc_n), is_causal=causal, pv_mode=pv,
                                                          strategy="gather", transport=transport, head_groups=2)
                    torch.cuda.synchronize()
                except Exception as e:  # symmetric memory may be unavailable on a box; NCCL must work
                    if transport != "peer":
                        raise
                    peer_error = repr(e)[:300]
                    continue
                res[(pv, causal, transport, gated)] = (out.cpu(), (whole_c if causal else whole_n).cpu())
        torch.save({"res": res, "peer_error": peer_error}, os.path.join(tmp, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_causal_and_gqa_sequence_sharding_match_unsharded_call(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp

    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        d = torch.load(os.path.join(tmp_path, f"r{r}.pt"))
        if d["peer_error"]:
            print("peer transport unavailable:", d["peer_error"])
        res = d["res"]
        for key, (a, b) in res.items():
            m = oracle.compare(a.float().numpy(), b.float().numpy())
            assert torch.equal(a, b), (key, m)
        assert all((pv, True, "nccl", "0") in res for pv in ("16bit", "fp8", "fp8_hilo"))
