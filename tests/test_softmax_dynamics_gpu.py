"""The fused kernel's online softmax on designed score landscapes (oracle/softmax_model.py), and batched GQA.

Random scores almost never move a row maximum by more than TAU within a 64-key step, so they leave the lazy rescale
(the warp vote, the early publish of P_{j-1}, the wait on PV_{j-1}, the rescale of O and of the tensor-core row sum L)
and the headroom p' -> 2^(KOFF + TAU) untested.  Each landscape here puts a rescale - or its absence - at a chosen step,
warp and query tile; tests/test_softmax_model_cpu.py proves on the CPU that it does.  Every landscape runs through
``fp8_attn_fwd`` in the three P modes, head-wise and token-wise, and through the 16-bit entry ``attn_fwd`` in bf16 and
fp16, against the fp64 oracle for O and for the LSE.

Bounds: O as in test_attention_gpu.py (row max-abs 0.02 of the row RMS; 0.30 for a single e4m3 P).  LSE: 2e-3 where
the row sum is accumulated from the fp32 p'; in the single-e4m3 P mode the row sum is that of the e4m3-rounded p'
(include/qattn.h), which moves the LSE by up to ln(1 + 2^-4), plus 2e-3 for the exponentials themselves.
"""
import pytest
import torch

import oracle
import quantum_attn
from oracle import softmax_model as sm
from quantumattention_b200 import _native

pytestmark = pytest.mark.gpu

PMODE = {"fp8": _native.QA_P_E4M3, "fp8_hilo": _native.QA_P_E4M3_HILO, "16bit": _native.QA_P_16BIT}
ROW_BOUND = {"fp8": 0.30, "fp8_hilo": 0.02, "16bit": 0.02}
LSE_BOUND = {"fp8": sm.e4m3_lse_bound(), "fp8_hilo": 2e-3, "16bit": 2e-3}


def oracle_out_lse(x, v, causal):
    """fp64 softmax(x * ln 2) @ v and its natural-log LSE; x [B,H,Sq,Skv] (log2 units), v [B,H,Skv,D]."""
    s = torch.from_numpy(x) * sm.LN2
    if causal:
        Sq, Skv = x.shape[-2:]
        s = s.masked_fill(torch.ones(Sq, Skv, dtype=torch.bool).triu(1), float("-inf"))
    return torch.softmax(s, -1) @ torch.from_numpy(v), torch.logsumexp(s, -1)


def check(out, lse, ref, ref_lse, mode, tag):
    m = oracle.compare(out.float().cpu().numpy(), ref.numpy())
    assert m["finite"] and m["cos_sim"] >= 0.999, (tag, m)
    assert m["max_abs_over_row_rms"] <= ROW_BOUND[mode], (tag, m)
    err = (lse.cpu().double() - ref_lse).abs().max().item()
    assert err <= LSE_BOUND[mode], (tag, err)
    return err


def run_fp8_entry(L, mode, causal, token):
    dev = "cuda"
    q8 = torch.from_numpy(L.q8).view(torch.float8_e4m3fn).to(dev)
    k8 = torch.from_numpy(L.k8).view(torch.float8_e4m3fn).to(dev)
    if mode == "16bit":
        v, sv = torch.from_numpy(L.dequant()[2]).to(torch.bfloat16).to(dev), None
    else:
        v, sv = torch.from_numpy(L.v8).view(torch.float8_e4m3fn).to(dev), torch.from_numpy(L.scale_v).to(dev)
    sq, sk = torch.from_numpy(L.scale_q).to(dev), torch.from_numpy(L.scale_k).to(dev)
    return _native.fp8_attn_fwd(q8, k8, v, sq, sk, sv, scale_mode=_native.QA_SCALE_TOKEN if token else _native.QA_SCALE_HEAD,
                                is_causal=causal, sm_scale=L.sm_scale, p_mode=PMODE[mode], out_dtype=torch.bfloat16,
                                return_lse=True)


def run_16bit_entry(L, dtype, causal):
    q, k, v = (torch.from_numpy(t).to(dtype).cuda() for t in L.dequant())
    return _native.attn_fwd(q, k, v, is_causal=causal, sm_scale=L.sm_scale, return_lse=True)


@pytest.mark.parametrize("fam", ["e4m3", "16bit"])
@pytest.mark.parametrize("case", sm.CASES, ids=[c.name for c in sm.CASES])
def test_landscape(case, fam):
    """e4m3 family: a single e4m3 P and e4m3 hi + lo P (TAU = 4); 16bit family: 16-bit P behind FP8 Q / K, and the
    16-bit entry in bf16 and fp16 (TAU = 8) - head-wise and token-wise scales for the FP8 entries."""
    tau, _ = sm.tau_koff(fam == "16bit")
    design = case.make(tau)
    head = sm.landscape(design, Sq=case.Sq, Skv=case.Skv, D=case.D, seed=1)
    tok = sm.landscape(design, Sq=case.Sq, Skv=case.Skv, D=case.D, token=True, seed=1)
    ref, ref_lse = oracle_out_lse(head.x, head.dequant()[2], case.causal)
    modes = ("fp8", "fp8_hilo") if fam == "e4m3" else ("16bit",)
    for mode in modes:
        for L, token in ((head, False), (tok, True)):
            out, lse = run_fp8_entry(L, mode, case.causal, token)
            check(out, lse, ref, ref_lse, mode, f"{case.name} {mode} {'token' if token else 'head'}")
    if fam == "16bit":
        for dtype in (torch.bfloat16, torch.float16):
            out, lse = run_16bit_entry(head, dtype, case.causal)
            assert out.dtype == dtype
            check(out, lse, ref, ref_lse, "16bit", f"{case.name} attn_fwd {dtype}")


@pytest.mark.parametrize("mode", ["16bit", "fp8_hilo"])
def test_long_landscape(mode):
    """Sq = 256 against Skv = 75 600 (the video shape's length: 1 182 steps, the last one 16 keys): six rescales in a
    row near the end, then one in the 16-key last step."""
    case = sm.LONG
    tau, _ = sm.tau_koff(mode == "16bit")
    L = sm.landscape(case.make(tau), Sq=case.Sq, Skv=case.Skv, D=case.D, seed=1)
    ref, ref_lse = oracle_out_lse(L.x, L.dequant()[2], False)
    out, lse = run_fp8_entry(L, mode, False, False)
    check(out, lse, ref, ref_lse, mode, f"long {mode}")


# ------------------------------------------------------------------------------------------------ batched GQA
def _gqa_inputs(B, Hq, Hkv, Sq, Skv, D, seed):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, Hq, Sq, D, generator=g)
    k = torch.randn(B, Hkv, Skv, D, generator=g)
    # (a different magnitude per (batch, kv head): V read from the wrong head cannot pass for the right one)
    v = torch.randn(B, Hkv, Skv, D, generator=g) * (1 + torch.arange(B * Hkv).reshape(B, Hkv, 1, 1))
    return (t.to(torch.bfloat16) for t in (q, k, v))


@pytest.mark.parametrize("shape", [(300, 1000, False), (520, 520, True)], ids=["300x1000", "520x520_causal"])
@pytest.mark.parametrize("heads", [(6, 2), (5, 1), (24, 8)], ids=["6_2", "5_1", "24_8"])
def test_batched_gqa(heads, shape):
    """B = 2 with Hq != Hkv, group sizes 3 and 5 too: the kv head of a query head (a float reciprocal in the kernel),
    the (b, kv head) index of the scales, and the public ``fp8_attn_func``'s own quantiser launches for Q and for K / V
    (token-wise: V apart, head-wise) - bit-identical to quantise-then-attend, as include/qattn.h states."""
    (Hq, Hkv), (Sq, Skv, causal) = heads, shape
    B, D, rep = 2, 128, Hq // Hkv
    q, k, v = _gqa_inputs(B, Hq, Hkv, Sq, Skv, D, seed=Hq * 100 + Sq)
    qc, kc, vc = q.cuda(), k.cuda(), v.cuda()
    mask = torch.ones(Sq, Skv, dtype=torch.bool).triu(1) if causal else None
    vr16 = v.double().repeat_interleave(rep, 1)
    for token in (False, True):
        sm_code = _native.QA_SCALE_TOKEN if token else _native.QA_SCALE_HEAD
        (q8,), (sq,) = _native.quantize_fp8([qc], sm_code)
        (k8,), (sk,) = _native.quantize_fp8([kc], sm_code)
        (v8,), (sv,) = _native.quantize_fp8([vc], _native.QA_SCALE_HEAD)
        qh = torch.from_numpy(oracle.dequantize(q8.view(torch.uint8).cpu().numpy(), sq.cpu().numpy())).double()
        kh = torch.from_numpy(oracle.dequantize(k8.view(torch.uint8).cpu().numpy(), sk.cpu().numpy())).double()
        vh8 = torch.from_numpy(oracle.dequantize(v8.view(torch.uint8).cpu().numpy(), sv.cpu().numpy())).double()
        s = (qh @ kh.repeat_interleave(rep, 1).transpose(-1, -2)) / D**0.5
        if causal:
            s = s.masked_fill(mask, float("-inf"))
        p, ref_lse = torch.softmax(s, -1), torch.logsumexp(s, -1)
        public = quantum_attn.fp8_token_wise_attn_func if token else quantum_attn.fp8_attn_func
        for mode in ("fp8", "fp8_hilo", "16bit"):
            tag = f"{heads} {shape} {'token' if token else 'head'} {mode}"
            vin, svin = (vc, None) if mode == "16bit" else (v8, sv)
            out, lse = _native.fp8_attn_fwd(q8, k8, vin, sq, sk, svin, scale_mode=sm_code, is_causal=causal,
                                            sm_scale=D**-0.5, p_mode=PMODE[mode], out_dtype=torch.bfloat16,
                                            return_lse=True)
            ref = p @ (vr16 if mode == "16bit" else vh8.repeat_interleave(rep, 1))
            check(out, lse, ref, ref_lse, mode, tag)
            with quantum_attn.config.patch({"attention.pv_mode": mode}):
                pub = public(qc, kc, vc, is_causal=causal)
            assert torch.equal(pub, out), tag
    # the 16-bit entry: same grouping, its own oracle on the unquantised inputs
    out, lse = _native.attn_fwd(qc, kc, vc, is_causal=causal, sm_scale=D**-0.5, return_lse=True)
    assert torch.equal(quantum_attn.attn_func(qc, kc, vc, is_causal=causal), out)
    s = (q.double() @ k.double().repeat_interleave(rep, 1).transpose(-1, -2)) / D**0.5
    if causal:
        s = s.masked_fill(mask, float("-inf"))
    check(out, lse, torch.softmax(s, -1) @ vr16, torch.logsumexp(s, -1), "16bit", f"{heads} {shape} attn_fwd")
