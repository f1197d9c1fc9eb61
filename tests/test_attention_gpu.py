"""Parity of the fused sm_100a attention kernel with the oracle (fp32/fp64 SDPA on the dequantised inputs).

Tolerances (BASELINE.json north_star): cosine similarity >= 0.999 for every mode; max-abs error <= 2e-2 x output RMS
is asserted row-wise for the modes whose arithmetic can meet it (16-bit P, e4m3 hi+lo P) - a single e4m3 P carries
3 mantissa bits and sits at ~0.15 x row-RMS (SURVEY.md Appendix A.5), so for "fp8" the bound asserted is the
reference's own gate, absolute RMSE < 1e-2 (tests/test_interface.py:57-59), plus a looser max-abs bound.
"""
import math
import os

import numpy as np
import pytest
import torch

import oracle
import quantum_attn
from quantumattention_b200 import _native
from conftest import bf16_from_bits

pytestmark = pytest.mark.gpu

PV = {"fp8": _native.QA_P_E4M3, "fp8_hilo": _native.QA_P_E4M3_HILO, "16bit": _native.QA_P_16BIT}
# max-abs error over the row RMS.  The north star's 2e-2 is asserted for the modes whose arithmetic can meet it; a single
# e4m3 P ("fp8", opt-in) carries 2^-4 relative steps per probability and is only held to a loose sanity bound.
ROW_BOUND = {"fp8": 0.30, "fp8_hilo": 0.02, "16bit": 0.02}


def run_native(q, k, v, *, causal, pv, mode="head-wise", scale=None, return_lse=False):
    """q,k,v: CPU 16-bit tensors. Returns (out_cpu_fp32, oracle_inputs dict)."""
    sm = _native.QA_SCALE_HEAD if mode == "head-wise" else _native.QA_SCALE_TOKEN
    qc, kc, vc = q.cuda(), k.cuda(), v.cuda()
    if q.shape[1] == k.shape[1]:
        (q8, k8), (sq, sk) = _native.quantize_fp8([qc, kc], sm)
    else:
        (q8,), (sq,) = _native.quantize_fp8([qc], sm)
        (k8,), (sk,) = _native.quantize_fp8([kc], sm)
    if pv == "16bit":
        v_in, sv = vc, None
    else:
        (v_in,), (sv,) = _native.quantize_fp8([vc], _native.QA_SCALE_HEAD)
    sm_scale = 1.0 / math.sqrt(q.shape[-1]) if scale is None else scale
    res = _native.fp8_attn_fwd(q8, k8, v_in, sq, sk, sv, scale_mode=sm, is_causal=causal, sm_scale=sm_scale,
                               p_mode=PV[pv], out_dtype=v.dtype, return_lse=return_lse)
    torch.cuda.synchronize()
    out, lse = (res if return_lse else (res, None))
    rep = q.shape[1] // k.shape[1]
    k8n = k8.view(torch.uint8).cpu().numpy().repeat(rep, axis=1)
    skn = sk.cpu().numpy().repeat(rep, axis=1)
    if pv == "16bit":
        vn, svn = v.float().numpy().repeat(rep, axis=1), None
    else:
        vn, svn = v_in.view(torch.uint8).cpu().numpy().repeat(rep, axis=1), sv.cpu().numpy().repeat(rep, axis=1)
    ref = oracle.fp8_attention_ref(q8.view(torch.uint8).cpu().numpy(), k8n, vn, sq.cpu().numpy(), skn,
                                   scale_v=svn, is_causal=causal, scale=scale)
    return out.float().cpu(), ref, lse


REL_RMSE_BOUND = {"fp8": 0.04, "fp8_hilo": 0.006, "16bit": 0.006}


def check(out, ref, pv, tag="", unit_scale=True, row_bound=None):
    m = oracle.compare(out.numpy(), ref.numpy())
    assert m["finite"], tag
    assert m["cos_sim"] >= 0.999, (tag, m)
    if unit_scale:  # randn inputs: the reference's own absolute gate applies (tests/test_interface.py:57-59)
        assert m["rmse"] < 1e-2, (tag, m)
    assert m["rmse_over_rms"] < REL_RMSE_BOUND[pv], (tag, m)
    assert m["max_abs_over_row_rms"] <= (ROW_BOUND[pv] if row_bound is None else row_bound), (tag, m)
    return m


@pytest.mark.parametrize("pv", ["fp8", "fp8_hilo", "16bit"])
@pytest.mark.parametrize("name", ["attn_d64_causal", "attn_d128", "attn_d256_causal"])
def test_golden_fixtures_from_reference(golden_dir, name, pv):
    """Same quantised inputs the reference saw; output vs the reference's own output (its gate: RMSE < 1e-2)."""
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    q8 = torch.from_numpy(g["q8"]).view(torch.float8_e4m3fn).cuda()
    k8 = torch.from_numpy(g["k8"]).view(torch.float8_e4m3fn).cuda()
    v = bf16_from_bits(g["v_bf16_bits"]).cuda()
    sq, sk = torch.from_numpy(g["scale_q"]).cuda(), torch.from_numpy(g["scale_k"]).cuda()
    causal = bool(g["causal"])
    if pv == "16bit":
        v_in, sv = v, None
    else:
        (v_in,), (sv,) = _native.quantize_fp8([v], _native.QA_SCALE_HEAD)
    out = _native.fp8_attn_fwd(q8, k8, v_in, sq, sk, sv, scale_mode=_native.QA_SCALE_HEAD, is_causal=causal,
                               sm_scale=1.0 / math.sqrt(q8.shape[-1]), p_mode=PV[pv], out_dtype=torch.bfloat16)
    out = out.float().cpu().numpy()
    ref_bf16 = bf16_from_bits(g["out_ref_bf16_bits"]).float().numpy()
    m = oracle.compare(out, ref_bf16)
    assert m["cos_sim"] >= 0.999 and m["rmse"] < 1e-2, m
    if pv == "16bit":  # same arithmetic as the reference kernel: agreement at bf16 resolution vs the fp32 statement
        m2 = oracle.compare(out, g["out_ref_fp32"])
        assert m2["max_abs_over_row_rms"] <= 0.02, m2


def test_golden_token_wise(golden_dir):
    g = np.load(os.path.join(golden_dir, "attn_d128_token.npz"))
    q8 = torch.from_numpy(g["q8"]).view(torch.float8_e4m3fn).cuda()
    k8 = torch.from_numpy(g["k8"]).view(torch.float8_e4m3fn).cuda()
    v = bf16_from_bits(g["v_bf16_bits"]).cuda()
    sq, sk = torch.from_numpy(g["scale_q"]).cuda(), torch.from_numpy(g["scale_k"]).cuda()
    out = _native.fp8_attn_fwd(q8, k8, v, sq, sk, None, scale_mode=_native.QA_SCALE_TOKEN, is_causal=False,
                               sm_scale=1.0 / math.sqrt(128), p_mode=PV["16bit"], out_dtype=torch.bfloat16)
    m = oracle.compare(out.float().cpu().numpy(), g["out_ref_fp32"])
    assert m["cos_sim"] >= 0.9999 and m["max_abs_over_row_rms"] <= 0.02, m


# C1 of BASELINE.json plus the reference's own test sweep shapes (tests/test_interface.py:62-84), scaled to H=2
@pytest.mark.parametrize("pv", ["fp8", "fp8_hilo", "16bit"])
@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("B,H,Sq,Skv,D", [
    (2, 8, 512, 512, 64),      # C1
    (1, 2, 1024, 1024, 128),
    (1, 2, 1000, 1000, 128),   # ragged
    (1, 2, 999, 999, 64),
    (1, 2, 1000, 1024, 128),   # Sq != Skv (causal: the top-left mask, as torch SDPA's is_causal)
    (1, 2, 1024, 1000, 256),
    (1, 2, 1000, 1000, 256),
    (1, 1, 1, 1, 128),         # degenerate
    (1, 1, 129, 3, 64),
    # where the per-tile step counts, the first masked step and the all-padding second query tile change
    (1, 2, 64, 64, 64),
    (1, 2, 65, 65, 128),
    (1, 2, 128, 128, 256),
    (1, 2, 129, 129, 64),
    (1, 2, 256, 256, 128),
    (1, 2, 257, 257, 256),
    (1, 2, 257, 65, 128),
    (1, 2, 1, 4097, 64),
])
def test_parity_sweep(B, H, Sq, Skv, D, causal, pv):
    q, k, v = oracle.make_qkv(B, H, Sq, Skv, D, seed=Sq + D)
    out, ref, _ = run_native(q, k, v, causal=causal, pv=pv)
    check(out, ref, pv, f"{(B, H, Sq, Skv, D, causal, pv)}")


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("pv", ["fp8", "16bit"])
def test_dtypes(dtype, pv):
    q, k, v = oracle.make_qkv(1, 2, 300, 300, 128, dtype=dtype, seed=11)
    out, ref, _ = run_native(q, k, v, causal=True, pv=pv)
    check(out, ref, pv)


@pytest.mark.parametrize("pv", ["fp8", "16bit"])
@pytest.mark.parametrize("causal", [False, True])
def test_token_wise_scales(pv, causal):
    q, k, v = oracle.make_qkv(1, 2, 700, 700, 128, seed=4, kind="outlier_channels")
    out, ref, _ = run_native(q, k, v, causal=causal, pv=pv, mode="token-wise")
    # heavy-tailed channels (exp(2 * randn) per channel): output rows are dominated by a few huge value channels, and the
    # bf16 rounding of those entries alone reaches 2.6e-2 of the row RMS (measured on B200); the 2e-2 bound is stated -
    # and asserted everywhere else - for the unit-scale shapes of BASELINE.json
    check(out, ref, pv, unit_scale=False, row_bound=0.03 if pv == "16bit" else None)


@pytest.mark.parametrize("S,D,causal,hq,hkv,pv", [
    (333, 64, False, 2, 2, "16bit"),     # Skv % 4 != 0: rows of scale_k are not 16-byte aligned (no bulk copy of the scales)
    (1030, 128, True, 2, 2, "16bit"),    # ragged, not a multiple of 4 either, several trips round the K / V ring
    (2052, 128, False, 4, 2, "16bit"),   # aligned rows + ragged tail (2052 = 16 * 128 + 4), GQA: scales of the kv head
    (1500, 256, True, 2, 2, "16bit"),
    (1500, 256, False, 2, 2, "fp8"),
    (2052, 64, True, 2, 1, "fp8"),
])
def test_token_wise_shapes(S, D, causal, hq, hkv, pv):
    """Per-token K scales travel to the softmax threads through shared memory (one bulk copy per K / V tile, or - when a
    row of scale_k is not 16-byte aligned - plain loads by the producer lane): every head dimension, ragged tails, ring
    wrap-around, GQA.  Semantics: inductor/kernels/attention.py:391-396,570-573 of the reference."""
    g = torch.Generator().manual_seed(S + D)
    q = torch.randn(1, hq, S, D, generator=g).to(torch.bfloat16)
    k = (torch.randn(1, hkv, S, D, generator=g) * torch.exp(torch.randn(1, hkv, S, 1, generator=g))).to(torch.bfloat16)
    v = torch.randn(1, hkv, S, D, generator=g).to(torch.bfloat16)
    out, ref, _ = run_native(q, k, v, causal=causal, pv=pv, mode="token-wise")
    check(out, ref, pv, tag=f"S{S} D{D}", unit_scale=False)


@pytest.mark.parametrize("kind", ["outlier_channels", "huge_token", "zero_head"])
def test_stress_inputs(kind):
    q, k, v = oracle.make_qkv(1, 2, 520, 520, 128, seed=6, kind=kind)
    out, ref, _ = run_native(q, k, v, causal=False, pv="16bit")
    m = oracle.compare(out.numpy(), ref.numpy())
    assert m["finite"] and m["cos_sim"] >= 0.999, m


def test_gqa_and_custom_scale_and_lse():
    g = torch.Generator().manual_seed(8)
    q = torch.randn(1, 8, 384, 128, generator=g).to(torch.bfloat16)
    k = torch.randn(1, 2, 384, 128, generator=g).to(torch.bfloat16)
    v = torch.randn(1, 2, 384, 128, generator=g).to(torch.bfloat16)
    out, ref, lse = run_native(q, k, v, causal=True, pv="16bit", scale=0.05, return_lse=True)
    check(out, ref, "16bit")
    # LSE against the oracle's scores
    (q8, ), (sq, ) = _native.quantize_fp8([q.cuda()], _native.QA_SCALE_HEAD)
    (k8, ), (sk, ) = _native.quantize_fp8([k.cuda()], _native.QA_SCALE_HEAD)
    qh = torch.from_numpy(oracle.dequantize(q8.view(torch.uint8).cpu().numpy(), sq.cpu().numpy())).double()
    kh = torch.from_numpy(oracle.dequantize(k8.view(torch.uint8).cpu().numpy(), sk.cpu().numpy())).double()
    s = (qh @ kh.repeat_interleave(4, 1).transpose(-1, -2)) * 0.05
    s = s.masked_fill(torch.ones(384, 384, dtype=torch.bool).triu(1), float("-inf"))
    assert torch.allclose(lse.cpu().double(), torch.logsumexp(s, -1), atol=2e-3)


def test_public_api_like_reference_test():
    """The reference's own correctness test, verbatim in spirit (tests/test_interface.py:31-59): fp8_attn_func vs
    torch FlashAttention on the UNQUANTISED inputs, RMSE < 1e-2; plus the eager composite as on-box comparator."""
    from torch.nn.attention import SDPBackend, sdpa_kernel

    torch.manual_seed(0)
    for (B, H, S, D, causal, dtype) in [(2, 8, 1024, 128, False, torch.bfloat16), (1, 16, 1000, 64, True, torch.float16),
                                        (1, 8, 1024, 256, True, torch.bfloat16)]:
        q = torch.randn(B, H, S, D, dtype=dtype, device="cuda")
        k = torch.randn(B, H, S, D, dtype=dtype, device="cuda")
        v = torch.randn(B, H, S, D, dtype=dtype, device="cuda")
        for pv in ("fp8", "fp8_hilo", "16bit"):
            with quantum_attn.config.patch({"attention.pv_mode": pv}):
                out = quantum_attn.fp8_attn_func(q, k, v, is_causal=causal)
            with sdpa_kernel(SDPBackend.FLASH_ATTENTION):
                fa = torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=causal)
            rmse = torch.sqrt(torch.nn.functional.mse_loss(out.float(), fa.float())).item()
            assert out.dtype == dtype and out.shape == q.shape and out.is_contiguous()
            assert rmse < 1e-2, (pv, rmse)
        with quantum_attn.config.patch({"attention.force_eager_fallback": True}):
            eager = quantum_attn.fp8_attn_func(q, k, v, is_causal=causal)
        with quantum_attn.config.patch({"attention.pv_mode": "16bit"}):
            ours = quantum_attn.fp8_attn_func(q, k, v, is_causal=causal)
        assert torch.sqrt(torch.nn.functional.mse_loss(ours.float(), eager.float())).item() < 3e-3
        tw = quantum_attn.fp8_token_wise_attn_func(q, k, v, is_causal=causal)
        assert torch.sqrt(torch.nn.functional.mse_loss(tw.float(), fa.float())).item() < 1e-2
        fb = quantum_attn.fp8_attn_func_with_fallback(q, k, v, is_causal=causal)
        assert torch.sqrt(torch.nn.functional.mse_loss(fb.float(), fa.float())).item() < 1e-2


def test_prequantized_inputs_and_errors():
    q, k, v = oracle.make_qkv(1, 2, 256, 256, 128, seed=3)
    qc, kc, vc = q.cuda(), k.cuda(), v.cuda()
    q8, sq = quantum_attn.dynamically_quantize_fp8(qc, reduction_dim=[2, 3])
    k8, sk = quantum_attn.dynamically_quantize_fp8(kc, reduction_dim=[2, 3])
    a = quantum_attn.fp8_attn_func(q8, k8, vc, scale_q=sq, scale_k=sk)
    b = quantum_attn.fp8_attn_func(qc, kc, vc)
    assert torch.equal(a, b)
    with pytest.raises(ValueError):
        quantum_attn.fp8_attn_func(qc, kc, vc, attn_mask=torch.ones(256, 256, device="cuda", dtype=torch.bool))
    with pytest.raises(ValueError):
        quantum_attn.fp8_attn_func(qc, kc, vc, dropout_p=0.1)
    with pytest.raises(ValueError):
        quantum_attn.fp8_attn_func(qc[..., :96], kc[..., :96], vc[..., :96])
    with pytest.raises(ValueError):
        quantum_attn.fp8_attn_func(qc, kc, vc, scale_q=sq, scale_k=sk)  # 16-bit q/k together with scales


@pytest.mark.parametrize("name", ["C2_flux", "C3_llama"])
def test_full_size_properties_and_oracle_on_2_heads_x_384_rows(name):
    """BASELINE configs at full size: the oracle only scores a slice - 2 heads x 384 rows (first / middle / last
    128), all keys - since it would take minutes otherwise;
    the rest is covered by size-independent properties: rows of softmax sum to one (V = 1 -> O = 1), and
    permuting the keys/values of a non-causal problem leaves O unchanged."""
    B, H, S, D, causal = oracle.CONFIGS[name]
    q, k, v = oracle.make_qkv(B, H, S, S, D, seed=0)
    qc, kc, vc = q.cuda(), k.cuda(), v.cuda()
    for pv in ("fp8", "16bit"):
        with quantum_attn.config.patch({"attention.pv_mode": pv}):
            out = quantum_attn.fp8_attn_func(qc, kc, vc, is_causal=causal)
            ones = quantum_attn.fp8_attn_func(qc, kc, torch.ones_like(vc), is_causal=causal)
            assert bool(torch.isfinite(out).all())
            # (single-e4m3 mode normalises by the tensor-core row sum of the SAME quantised weights that multiply V,
            # so the rows sum to one as tightly as in the 16-bit mode)
            assert (ones.float() - 1.0).abs().max().item() < 0.01
            if not causal:
                perm = torch.randperm(S, generator=torch.Generator().manual_seed(1)).cuda()
                outp = quantum_attn.fp8_attn_func(qc, kc[:, :, perm], vc[:, :, perm], is_causal=False)
                m = oracle.compare(outp.float().cpu().numpy(), out.float().cpu().numpy())
                # two runs that round P to e4m3 in different key orders differ by ~sqrt(2) x the single-run error
                assert m["cos_sim"] > (0.999 if pv == "fp8" else 0.99995), m
        # oracle on a slice: 2 heads x 3 row blocks (first, middle, last rows)
        (q8, k8), (sq, sk) = _native.quantize_fp8([qc, kc], _native.QA_SCALE_HEAD)
        heads = [0, H - 1]
        rows = torch.cat([torch.arange(0, 128), torch.arange(S // 2 - 64, S // 2 + 64), torch.arange(S - 128, S)])
        if pv == "16bit":
            vh = v[:, heads].float().numpy()
        else:
            (v8,), (sv,) = _native.quantize_fp8([vc], _native.QA_SCALE_HEAD)
            vh = oracle.dequantize(v8.view(torch.uint8).cpu().numpy()[:, heads], sv.cpu().numpy()[:, heads])
        qh = oracle.dequantize(q8.view(torch.uint8).cpu().numpy()[:, heads], sq.cpu().numpy()[:, heads])
        kh = oracle.dequantize(k8.view(torch.uint8).cpu().numpy()[:, heads], sk.cpu().numpy()[:, heads])
        qh, kh, vh = (torch.from_numpy(x).double() for x in (qh, kh, vh))
        sc = (qh[:, :, rows] @ kh.transpose(-1, -2)) / math.sqrt(D)
        if causal:
            sc = sc.masked_fill(torch.arange(S)[None, :] > rows[:, None], float("-inf"))
        ref = torch.softmax(sc, -1) @ vh
        m = oracle.compare(out[:, heads][:, :, rows].float().cpu().numpy(), ref.numpy())
        assert m["cos_sim"] >= 0.999 and m["max_abs_over_row_rms"] <= ROW_BOUND[pv], (pv, m)


@pytest.mark.parametrize("pv", ["16bit", "fp8_hilo", "fp8"])
def test_full_size_video_shape_oracle_on_2_heads_x_384_rows(pv):
    """C4 (B1 H24 S75600 D128, ragged: 75600 = 590 * 128 + 80) on one GPU at full size, each P mode against ITS oracle
    (16-bit V for "16bit", dequantised e4m3 V for the FP8 modes) with its own bound: finite output, rows of softmax
    sum to one, and the fp64 oracle on a slice (first / middle / last 128 rows of the first and last head, all keys)."""
    B, H, S, D, causal = oracle.CONFIGS["C4_video"]
    g = torch.Generator(device="cuda").manual_seed(4)
    qc, kc, vc = (torch.randn((B, H, S, D), device="cuda", dtype=torch.bfloat16, generator=g) for _ in range(3))
    with quantum_attn.config.patch({"attention.pv_mode": pv}):
        out = quantum_attn.fp8_attn_func(qc, kc, vc, is_causal=causal)
        assert out.shape == qc.shape and bool(torch.isfinite(out).all())
        ones = quantum_attn.fp8_attn_func(qc, kc, torch.ones_like(vc), is_causal=causal)
        assert (ones.float() - 1.0).abs().max().item() < 0.01
        del ones
    heads = [0, H - 1]
    rows = torch.cat([torch.arange(0, 128), torch.arange(S // 2 - 64, S // 2 + 64), torch.arange(S - 128, S)])
    (q8, k8), (sq, sk) = _native.quantize_fp8([qc[:, heads], kc[:, heads]], _native.QA_SCALE_HEAD)
    deq = lambda x8, sc: torch.from_numpy(oracle.dequantize(x8.view(torch.uint8).cpu().numpy(), sc.cpu().numpy())).double()
    qh, kh = deq(q8, sq)[:, :, rows], deq(k8, sk)
    if pv == "16bit":
        vh = vc[:, heads].double().cpu()
    else:
        (v8,), (sv,) = _native.quantize_fp8([vc[:, heads]], _native.QA_SCALE_HEAD)
        vh = deq(v8, sv)
    ref = torch.softmax((qh @ kh.transpose(-1, -2)) / math.sqrt(D), -1) @ vh
    m = oracle.compare(out[:, heads][:, :, rows.cuda()].float().cpu().numpy(), ref.numpy())
    assert m["cos_sim"] >= 0.999 and m["max_abs_over_row_rms"] <= ROW_BOUND[pv], (pv, m)
