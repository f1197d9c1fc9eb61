"""Parity of the 16-bit path (`attn_func` / op `quantum_attn::attention_forward` / C ABI `qa_attn_fwd`) with the oracle:
fp64 SDPA on the same bf16 / fp16 inputs (reference definition: src/quantum_attn/ops.py:15-28), the fixtures recorded
from the reference, and the reference's own test (tests/test_interface.py:62-73: RMSE < 1e-2 vs FlashAttention).

Tolerances: cosine similarity >= 0.9999, max-abs error <= 2e-2 x row RMS (BASELINE.json north_star), RMSE < 1e-2.
"""
import math
import os

import numpy as np
import pytest
import torch

import oracle
import quantum_attn
from quantumattention_b200 import _native
from conftest import f16_from_bits

pytestmark = pytest.mark.gpu


def check(out, ref, tag=""):
    m = oracle.compare(out.float().cpu().numpy(), ref.numpy() if torch.is_tensor(ref) else ref)
    assert m["finite"], tag
    assert m["cos_sim"] >= 0.9999, (tag, m)
    assert m["rmse"] < 1e-2, (tag, m)
    assert m["max_abs_over_row_rms"] <= 0.02, (tag, m)
    return m


@pytest.mark.parametrize("name", ["attn16_d64_causal", "attn16_d128", "attn16_d128_fp16_causal", "attn16_d256_causal"])
def test_golden_fixtures_from_reference(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    fp16 = bool(g["fp16"])
    q, k, v = (f16_from_bits(g[n], fp16).cuda() for n in ("q_bits", "k_bits", "v_bits"))
    out = _native.attn_fwd(q, k, v, is_causal=bool(g["causal"]), sm_scale=1.0 / math.sqrt(q.shape[-1]))
    assert out.dtype == q.dtype and out.shape == q.shape
    check(out, g["out_ref_fp32"], name)
    # and against the reference's own 16-bit arithmetic: two 16-bit roundings apart
    m = oracle.compare(out.float().cpu().numpy(), f16_from_bits(g["out_ref_16_bits"], fp16).float().numpy())
    assert m["cos_sim"] >= 0.9999 and m["rmse"] < 1e-2, m


@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("B,H,Sq,Skv,D", [
    (2, 8, 512, 512, 64),      # C1
    (1, 2, 1024, 1024, 128),
    (1, 2, 999, 999, 128),     # ragged (the reference's 16-bit sweep uses 999, tests/test_interface.py:64-65)
    (1, 2, 999, 999, 64),
    (1, 2, 999, 1024, 128),    # Sq != Skv (causal: the top-left mask, as torch SDPA's is_causal)
    (1, 2, 1024, 999, 256),
    (1, 2, 999, 999, 256),
    (1, 2, 2100, 2100, 256),   # D = 256 runs a one-stage K/V ring: many tiles through the same slot
    (1, 1, 1, 1, 128),         # degenerate
    (1, 1, 129, 3, 64),
    # where the per-tile step counts, the first masked step and the all-padding second query tile change
    (1, 2, 64, 64, 128),
    (1, 2, 65, 65, 256),
    (1, 2, 128, 128, 64),
    (1, 2, 129, 129, 128),
    (1, 2, 256, 256, 256),
    (1, 2, 257, 257, 64),
    (1, 2, 257, 65, 256),
    (1, 2, 1, 4097, 128),
])
def test_parity_sweep(B, H, Sq, Skv, D, causal):
    q, k, v = oracle.make_qkv(B, H, Sq, Skv, D, seed=Sq + D)
    out = _native.attn_fwd(q.cuda(), k.cuda(), v.cuda(), is_causal=causal, sm_scale=1.0 / math.sqrt(D))
    check(out, oracle.sdpa_ref(q, k, v, is_causal=causal), f"{(B, H, Sq, Skv, D, causal)}")


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("kind", ["randn", "outlier_channels", "zero_head"])
def test_dtypes_and_stress_inputs(dtype, kind):
    q, k, v = oracle.make_qkv(1, 2, 520, 520, 128, dtype=dtype, seed=6, kind=kind)
    out = _native.attn_fwd(q.cuda(), k.cuda(), v.cuda(), is_causal=True, sm_scale=1.0 / math.sqrt(128))
    ref = oracle.sdpa_ref(q, k, v, is_causal=True)
    m = oracle.compare(out.float().cpu().numpy(), ref.numpy())
    assert out.dtype == dtype and m["finite"] and m["cos_sim"] >= 0.9999 and m["max_abs_over_row_rms"] <= 0.03, m


def test_gqa_custom_scale_and_lse():
    g = torch.Generator().manual_seed(8)
    q = torch.randn(1, 8, 384, 128, generator=g).to(torch.bfloat16)
    k = torch.randn(1, 2, 384, 128, generator=g).to(torch.bfloat16)
    v = torch.randn(1, 2, 384, 128, generator=g).to(torch.bfloat16)
    out, lse = _native.attn_fwd(q.cuda(), k.cuda(), v.cuda(), is_causal=True, sm_scale=0.05, return_lse=True)
    kr, vr = k.repeat_interleave(4, 1), v.repeat_interleave(4, 1)
    check(out, oracle.sdpa_ref(q, kr, vr, is_causal=True, scale=0.05))
    s = (q.double() @ kr.double().transpose(-1, -2)) * 0.05
    s = s.masked_fill(torch.ones(384, 384, dtype=torch.bool).triu(1), float("-inf"))
    assert torch.allclose(lse.cpu().double(), torch.logsumexp(s, -1), atol=2e-3)


def test_public_api_like_reference_test():
    """tests/test_interface.py:62-73 in spirit: attn_func vs torch FlashAttention, RMSE < 1e-2; output contract; the op;
    the with_fallback composite; the eager definition as on-box comparator; error behaviour."""
    from torch.nn.attention import SDPBackend, sdpa_kernel

    torch.manual_seed(0)
    for (B, H, Sq, Skv, D, causal, dtype) in [(2, 8, 1024, 1024, 128, False, torch.bfloat16),
                                              (1, 16, 999, 999, 64, True, torch.float16),
                                              (1, 8, 1024, 999, 256, False, torch.bfloat16),
                                              (2, 8, 999, 999, 256, True, torch.float16)]:
        q = torch.randn(B, H, Sq, D, dtype=dtype, device="cuda")
        k = torch.randn(B, H, Skv, D, dtype=dtype, device="cuda")
        v = torch.randn(B, H, Skv, D, dtype=dtype, device="cuda")
        with sdpa_kernel(SDPBackend.FLASH_ATTENTION):
            fa = torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=causal)
        out = quantum_attn.attn_func(q, k, v, is_causal=causal)
        assert out.dtype == dtype and out.shape == q.shape and out.is_contiguous()
        rmse = lambda a, b: torch.sqrt(torch.nn.functional.mse_loss(a.float(), b.float())).item()  # noqa: E731
        assert rmse(out, fa) < 1e-2
        assert torch.equal(torch.ops.quantum_attn.attention_forward(q, k, v, is_causal=causal), out)
        assert torch.equal(quantum_attn.attn_func_with_fallback(q, k, v, is_causal=causal), out)
        with quantum_attn.config.patch({"attention.force_eager_fallback": True}):
            eager = quantum_attn.attn_func(q, k, v, is_causal=causal)
        assert rmse(out, eager) < 3e-3
        # strided views are accepted (made dense on the way in, as the reference does, tk/attention.py:419-421)
        qt = q.transpose(1, 2).contiguous().transpose(1, 2)
        assert torch.equal(quantum_attn.attn_func(qt, k, v, is_causal=causal), out)
    with pytest.raises(ValueError):
        quantum_attn.attn_func(q, k, v, attn_mask=torch.ones(999, 999, device="cuda", dtype=torch.bool))
    with pytest.raises(ValueError):
        quantum_attn.attn_func(q, k, v, dropout_p=0.1)
    with pytest.raises(ValueError):
        quantum_attn.attn_func(q, k.to(torch.bfloat16), v)
    with pytest.raises(ValueError):
        quantum_attn.attn_func(q[..., :96], k[..., :96], v[..., :96])


@pytest.mark.parametrize("name", ["C2_flux", "C3_llama"])
def test_full_size_properties(name):
    """BASELINE shapes at full size: rows of softmax sum to one (V = 1 -> O = 1), key permutation invariance
    (non-causal), and the oracle on a slice of heads x rows."""
    B, H, S, D, causal = oracle.CONFIGS[name]
    q, k, v = oracle.make_qkv(B, H, S, S, D, seed=0)
    qc, kc, vc = q.cuda(), k.cuda(), v.cuda()
    out = quantum_attn.attn_func(qc, kc, vc, is_causal=causal)
    ones = quantum_attn.attn_func(qc, kc, torch.ones_like(vc), is_causal=causal)
    assert bool(torch.isfinite(out).all())
    assert (ones.float() - 1.0).abs().max().item() < 0.01
    if not causal:
        perm = torch.randperm(S, generator=torch.Generator().manual_seed(1)).cuda()
        outp = quantum_attn.attn_func(qc, kc[:, :, perm], vc[:, :, perm], is_causal=False)
        m = oracle.compare(outp.float().cpu().numpy(), out.float().cpu().numpy())
        assert m["cos_sim"] > 0.99995, m
    heads = [0, H - 1]
    rows = torch.cat([torch.arange(0, 128), torch.arange(S // 2 - 64, S // 2 + 64), torch.arange(S - 128, S)])
    qh, kh, vh = (x[:, heads].double() for x in (q, k, v))
    sc = (qh[:, :, rows] @ kh.transpose(-1, -2)) / math.sqrt(D)
    if causal:
        sc = sc.masked_fill(torch.arange(S)[None, :] > rows[:, None], float("-inf"))
    ref = torch.softmax(sc, -1) @ vh
    m = oracle.compare(out[:, heads][:, :, rows].float().cpu().numpy(), ref.numpy())
    assert m["cos_sim"] >= 0.9999 and m["max_abs_over_row_rms"] <= 0.02, m
