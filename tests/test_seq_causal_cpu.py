"""Causal and GQA sequence sharding, host side, on CPU: the zig-zag layout, the gather strategy's call sequence under
gloo with world sizes 2 and 3 (kernels replaced by an fp64 oracle through the backend hook), and the C ABI's checks
of the causal mode.  The kernels themselves: tests/test_bottom_right_gpu.py; the NCCL / peer transports on two GPUs:
tests/test_seq_causal_gpu.py."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
from quantumattention_b200 import _native, parallel


class CausalOracleBackend:
    """parallel.NativeBackend's interface on fp64 CPU arithmetic, with the causal modes of the C ABI and GQA (kv head =
    q head // (Hq / Hkv)).  Records (q shape, k shape, causal) of every attend."""

    def __init__(self):
        self.calls = []

    def local_scales(self, tensors):
        return [torch.from_numpy(oracle.head_scales(t.float().numpy())) for t in tensors]

    def quantize(self, tensors, scales, outs=None):
        return [torch.from_numpy(oracle.quantize_with_scale(t.float().numpy(), s.numpy())).view(torch.float8_e4m3fn)
                for t, s in zip(tensors, scales)]

    def attend(self, q8, k8, v, sq, sk, sv, sm_scale, p_mode, out_dtype, out=None, return_lse=True, causal=0):
        self.calls.append((tuple(q8.shape), tuple(k8.shape), causal))
        deq = lambda x8, s: torch.from_numpy(oracle.dequantize(x8.contiguous().view(torch.uint8).numpy(),  # noqa: E731
                                                               s.contiguous().numpy())).double()
        q, k = deq(q8, sq), deq(k8, sk)
        vv = v.double() if sv is None else deq(v, sv)
        g = q.shape[1] // k.shape[1]
        k, vv = k.repeat_interleave(g, 1), vv.repeat_interleave(g, 1)
        s = (q @ k.transpose(-1, -2)) * sm_scale
        Sq, Skv = s.shape[-2:]
        if causal:
            off = 0 if causal == _native.QA_CAUSAL_TOP_LEFT else Skv - Sq
            s = s.masked_fill(torch.ones(Sq, Skv, dtype=torch.bool).triu(1 + off), float("-inf"))
        o = (torch.softmax(s, -1) @ vv).to(out_dtype)
        if out is not None:
            out.copy_(o)
            o = out
        return (o, torch.logsumexp(s, -1).float()) if return_lse else o


def full_causal_ref(q, k, v, pv):
    """The unsharded call: head-wise quantisation of the whole sequence, fp64 top-left causal attention (GQA by
    repeating the quantised K / V heads)."""
    g = q.shape[1] // k.shape[1]
    q8, sq = oracle.quantize_fp8(q.float().numpy(), "head-wise")
    k8, sk = oracle.quantize_fp8(k.float().numpy(), "head-wise")
    rep = lambda a: np.repeat(a, g, axis=1)  # noqa: E731
    if pv == "16bit":
        return oracle.fp8_attention_ref(q8, rep(k8), rep(v.float().numpy()), sq, rep(sk), is_causal=True)
    v8, sv = oracle.quantize_fp8(v.float().numpy(), "head-wise")
    return oracle.fp8_attention_ref(q8, rep(k8), rep(v8), sq, rep(sk), scale_v=rep(sv), is_causal=True)


def make_problem(world, c, Hq, Hkv, D=64):
    S = 2 * world * c
    g = torch.Generator().manual_seed(7 * world + Hq)
    q, k, v = (torch.randn(1, h, S, D, generator=g).to(torch.bfloat16) for h in (Hq, Hkv, Hkv))
    # shards with different amax, so that the MAX all-reduce of the scales matters
    return q, k * torch.linspace(0.5, 2.0, S).view(1, 1, -1, 1).to(k.dtype), v


def test_zigzag_round_trip_and_layout():
    x = torch.arange(2 * 24).view(1, 2, 24, 1)
    for world in (1, 2, 3, 4):
        shards = [parallel.zigzag_shard(x, world, r) for r in range(world)]
        assert torch.equal(parallel.zigzag_unshard(shards), x)
        c = 24 // (2 * world)
        for r, t in enumerate(shards):  # chunk r, then chunk 2N-1-r
            assert t[0, 0, :, 0].tolist() == list(range(r * c, (r + 1) * c)) + \
                list(range((2 * world - 1 - r) * c, (2 * world - r) * c))
    with pytest.raises(ValueError, match="multiple of 2"):
        parallel.zigzag_shard(x[:, :, :22], 4, 0)
    with pytest.raises(ValueError):
        parallel.zigzag_shard(x, 2, 2)


def test_one_rank_causal_is_the_plain_top_left_call():
    q, k, v = make_problem(1, 40, 4, 2)
    for pv in ("16bit", "fp8"):
        be = CausalOracleBackend()
        out = parallel.ring_fp8_attention(q, k, v, is_causal=True, backend=be, pv_mode=pv)
        assert be.calls == [((1, 4, 80, 64), (1, 2, 80, 64), _native.QA_CAUSAL_TOP_LEFT)]
        m = oracle.compare(out.float().numpy(), full_causal_ref(q, k, v, pv).numpy())
        assert m["cos_sim"] > 0.99999 and m["max_abs_over_row_rms"] < 2e-2, (pv, m)


def test_causal_ring_and_odd_shards_are_rejected():
    q, k, v = make_problem(1, 40, 2, 2)
    with pytest.raises(ValueError, match="non-causal only"):
        parallel.ring_fp8_attention(q, k, v, is_causal=True, strategy="ring", backend=CausalOracleBackend())
    with pytest.raises(ValueError, match="no GQA"):
        parallel.ring_fp8_attention(q, k[:, :1], v[:, :1], strategy="ring", backend=CausalOracleBackend())
    with pytest.raises(ValueError, match="multiple of Hkv"):
        parallel.ring_fp8_attention(q[:, :1], k, v, strategy="gather", backend=CausalOracleBackend())


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


CASES = [(4, 2), (2, 2)]  # (Hq, Hkv): GQA and MHA
C = 48  # chunk: not a multiple of the kernel's 64-key steps, so the diagonal offsets are not either


def _worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = {}
        for Hq, Hkv in CASES:
            q, k, v = make_problem(world, C, Hq, Hkv)
            loc = [parallel.zigzag_shard(t, world, rank) for t in (q, k, v)]
            for pv in ("16bit", "fp8"):
                be = CausalOracleBackend()
                out = parallel.ring_fp8_attention(*loc, is_causal=True, backend=be, strategy="gather", pv_mode=pv,
                                                  head_groups=Hkv)
                g = Hq // Hkv
                # per head group (one kv head here) two launches: chunk r over (r + 1) c keys, chunk 2N-1-r over
                # (2N - r) c keys, both with the diagonal at the last key
                want = [((1, g, C, 64), (1, 1, (rank + 1) * C, 64), _native.QA_CAUSAL_BOTTOM_RIGHT),
                        ((1, g, C, 64), (1, 1, (2 * world - rank) * C, 64), _native.QA_CAUSAL_BOTTOM_RIGHT)] * Hkv
                assert be.calls == want, be.calls
                # non-causal GQA through the same gather: one launch per group over all keys
                be2 = CausalOracleBackend()
                out_nc = parallel.ring_fp8_attention(*loc, backend=be2, strategy="gather", pv_mode=pv, head_groups=Hkv)
                assert be2.calls == [((1, g, 2 * C, 64), (1, 1, 2 * world * C, 64), 0)] * Hkv
                res[(Hq, Hkv, pv)] = (out, out_nc)
        torch.save(res, os.path.join(tmp, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_causal_gather_matches_unsharded_oracle(world, tmp_path):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    per_rank = [torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in range(world)]
    for Hq, Hkv in CASES:
        q, k, v = make_problem(world, C, Hq, Hkv)
        for pv in ("16bit", "fp8"):
            got = parallel.zigzag_unshard([d[(Hq, Hkv, pv)][0] for d in per_rank])
            m = oracle.compare(got.float().numpy(), full_causal_ref(q, k, v, pv).numpy())
            assert m["finite"] and m["cos_sim"] > 0.99999 and m["max_abs_over_row_rms"] < 2e-2, (Hq, Hkv, pv, m)
            # non-causal: the zig-zag shards are just another permutation of the queries against all keys
            g = Hq // Hkv
            q8, sq = oracle.quantize_fp8(q.float().numpy(), "head-wise")
            k8, sk = oracle.quantize_fp8(k.float().numpy(), "head-wise")
            rep = lambda a: np.repeat(a, g, axis=1)  # noqa: E731
            if pv == "16bit":
                ref_nc = oracle.fp8_attention_ref(q8, rep(k8), rep(v.float().numpy()), sq, rep(sk))
            else:
                v8, sv = oracle.quantize_fp8(v.float().numpy(), "head-wise")
                ref_nc = oracle.fp8_attention_ref(q8, rep(k8), rep(v8), sq, rep(sk), scale_v=rep(sv))
            got_nc = parallel.zigzag_unshard([d[(Hq, Hkv, pv)][1] for d in per_rank])
            m = oracle.compare(got_nc.float().numpy(), ref_nc.numpy())
            assert m["finite"] and m["cos_sim"] > 0.99999 and m["max_abs_over_row_rms"] < 2e-2, (Hq, Hkv, pv, m)


def test_causal_mode_is_checked_at_the_boundary():
    lib = _native.load()
    # (fake pointers: aligned as the header asks; the checks come before any device access)
    args = lambda Sq, Skv, causal: (16, 16, 16, 2, None, None, None, 16, 16, 16, 0, 32, 0, None, 1, 2, 2, Sq, Skv, 64,  # noqa: E731
                                    causal, 0.125, 2)
    rc = lib.qa_fp8_attn_fwd(*args(9, 8, _native.QA_CAUSAL_BOTTOM_RIGHT), None)
    assert rc == -1 and b"Sq <= Skv" in lib.qa_last_error()
    for bad in (3, -1, 255):
        rc = lib.qa_fp8_attn_fwd(*args(8, 8, bad), None)
        assert rc == -1 and b"causal must be" in lib.qa_last_error()
    rc = lib.qa_attn_fwd(16, 16, 16, 0, None, None, None, 32, None, 1, 2, 2, 9, 8, 64, _native.QA_CAUSAL_BOTTOM_RIGHT,
                         0.125, None)
    assert rc == -1 and b"Sq <= Skv" in lib.qa_last_error()
    rc = lib.qa_attn_fwd(16, 16, 16, 0, None, None, None, 32, None, 1, 2, 2, 8, 8, 64, 3, 0.125, None)
    assert rc == -1 and b"causal must be" in lib.qa_last_error()
    # the gated launch does not take the bottom-right mode: QA_ERR_UNSUPPORTED
    rc = lib.qa_fp8_attn_fwd_gated(*args(8, 8, _native.QA_CAUSAL_BOTTOM_RIGHT), 16, 1, 1, None)
    assert rc == -4 and b"BOTTOM_RIGHT" in lib.qa_last_error()
    # the binding turns QA_ERR_INVALID into ValueError
    with pytest.raises(ValueError, match="Sq <= Skv"):
        _native._check(lib.qa_fp8_attn_fwd(*args(9, 8, _native.QA_CAUSAL_BOTTOM_RIGHT), None), "qa_fp8_attn_fwd")
    assert _native.ABI_VERSION == lib.qa_abi_version() == 7
