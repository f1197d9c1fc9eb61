"""Causal attention with Sq != Skv: the top-left mask of torch SDPA's ``is_causal`` on rectangular problems, in every
kernel entry point.

Row i of a causal problem sees keys 0 .. min(i, Skv - 1).  With Sq > Skv the rows from Skv on see every key and are
masked by the ragged tail alone; with Sq < Skv a query tile stops at its diagonal, long before the last key.  The
kernel's per-tile step counts (``nst0`` / ``nst1``), first masked step (``j_mask``) and last visible column (``lim``)
each take a ``min`` with Skv that only a rectangular problem can resolve the other way (attn_fwd_kernel.cuh).

* oracle parity: fp64 softmax on the inputs as the kernel sees them, O and the LSE, for ``fp8_attn_fwd`` in the three
  P modes with head-wise and token-wise scales and for ``attn_fwd`` in bf16 and fp16, both directions, D 64 / 128 / 256,
  batched GQA; the public functions give the same bits as the entry they call;
* exact structure: a rectangular launch reproduces, bit for bit, the square causal launch on the keys (Sq < Skv) or
  on the query rows (Sq > Skv) the two share, and the non-causal launch on the rows past Skv;
* designed softmax landscapes (oracle/softmax_model.py: RECT_CASES) whose dominant keys lie past every row's diagonal,
  or rescale only the rows past a tile that stops early;
* the public API against its eager definition (aten SDPA, MATH backend), and a check that the bounds used here tell the
  top-left mask from the bottom-right one of KV-cache decoding.

Bounds: O as in test_attention_gpu.py (FP8 entry) and test_attention16_gpu.py (16-bit entry); the LSE as in
test_softmax_dynamics_gpu.py.
"""
import collections

import pytest
import torch

import oracle
import quantum_attn
from oracle import softmax_model as sm
from quantumattention_b200 import _native
from test_attention_gpu import REL_RMSE_BOUND, ROW_BOUND
from test_softmax_dynamics_gpu import LSE_BOUND, PMODE, oracle_out_lse, run_16bit_entry, run_fp8_entry
from test_softmax_dynamics_gpu import check as check_landscape

pytestmark = pytest.mark.gpu

HEAD, TOKEN = _native.QA_SCALE_HEAD, _native.QA_SCALE_TOKEN
BF16, FP16 = torch.bfloat16, torch.float16


def top_left(Sq, Skv):
    """True where a causal row may not look: key > row."""
    return torch.ones(Sq, Skv, dtype=torch.bool).triu(1)


def bottom_right(Sq, Skv):
    """The KV-cache alignment, for contrast: key > row + Skv - Sq (rows below Sq - Skv see no key)."""
    return torch.ones(Sq, Skv, dtype=torch.bool).triu(Skv - Sq + 1)


def probs(q, k, sm_scale, mask):
    """fp64 softmax(q k^T * sm_scale) under ``mask`` and its natural-log LSE; each K head serves Hq / Hkv query heads.
    A row that sees no key gets P = 0 (LSE -inf)."""
    s = (q.double() @ k.double().repeat_interleave(q.shape[1] // k.shape[1], 1).transpose(-1, -2)) * sm_scale
    s = s.masked_fill(mask, float("-inf"))
    lse = torch.logsumexp(s, -1)
    return torch.exp(s - lse[..., None]).nan_to_num(0.0), lse


def pv(p, v):
    return p @ v.double().repeat_interleave(p.shape[1] // v.shape[1], 1)


def deq(x8, s):
    return torch.from_numpy(oracle.dequantize(x8.view(torch.uint8).cpu().numpy(), s.cpu().numpy())).double()


def row_error(out, ref):
    """Largest |out - ref| over the RMS of its row of ``ref``, net of the output's own rounding: half an ulp of each
    element in the output dtype.  A row that sees few keys can hold an element several times its RMS, and rounding
    that element to bf16 moves it by up to 2^-9 of its magnitude - by itself close to 2e-2 of the row RMS.  (2100 x
    1030 at D 256, token-wise, 16-bit P: 0.0203 of the row RMS, 0.0078 of the 0.0079 error being the rounding of an
    element in [2, 4), measured on an NVIDIA B200 at a 1000 W power limit.)"""
    o = out.cpu().double()
    half_ulp = torch.ldexp(torch.full_like(o, torch.finfo(out.dtype).eps / 4), torch.frexp(o)[1]) * (o != 0)
    row_rms = ref.pow(2).mean(-1, keepdim=True).sqrt()
    return (((o - ref).abs() - half_ulp).clamp(min=0) / row_rms).max().item()


def check(out, lse, ref, ref_lse, mode, tag, entry16=False):
    """O: cosine, absolute and relative RMSE, row max-abs (``row_error``); the LSE to LSE_BOUND.  ``entry16``: the
    16-bit entry's tighter cosine (test_attention16_gpu.py)."""
    m = oracle.compare(out.float().cpu().numpy(), ref.numpy())
    assert m["finite"] and m["cos_sim"] >= (0.9999 if entry16 else 0.999), (tag, m)
    assert m["rmse"] < 1e-2 and m["rmse_over_rms"] < REL_RMSE_BOUND[mode], (tag, m)
    assert row_error(out, ref) <= ROW_BOUND[mode], (tag, row_error(out, ref), m)
    err = (lse.cpu().double() - ref_lse).abs().max().item()
    assert err <= LSE_BOUND[mode], (tag, err)
    return m


def make_inputs(B, Hq, Hkv, Sq, Skv, D, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, Hq, Sq, D, generator=g), torch.randn(B, Hkv, Skv, D, generator=g),
            torch.randn(B, Hkv, Skv, D, generator=g))


Entry = collections.namedtuple("Entry", "tag mode run q k v dtype public")


def entries(q, k, v):
    """Every kernel entry on fp32 CPU inputs.  ``run(nq, nk, causal)`` launches on Q[:, :, :nq] and K / V[:, :, :nk]:
    slices of the same quantised tensors and scales, so launches of different shapes see the same bytes.  ``q`` / ``k``
    / ``v``: fp64 Q, K, V as the entry reads them; ``public(causal)``: the public function that runs the entry in one
    call on the whole problem (quantiser included)."""
    sm_scale = q.shape[-1] ** -0.5
    qc, kc, vc = (t.to(BF16).cuda() for t in (q, k, v))
    (v8,), (sv,) = _native.quantize_fp8([vc], HEAD)
    for token in (False, True):
        code = TOKEN if token else HEAD
        (q8,), (sq,) = _native.quantize_fp8([qc], code)
        (k8,), (sk,) = _native.quantize_fp8([kc], code)
        fn = quantum_attn.fp8_token_wise_attn_func if token else quantum_attn.fp8_attn_func
        for mode in PMODE:
            vin, svin = (vc, None) if mode == "16bit" else (v8, sv)

            def run(nq, nk, causal, q8=q8, k8=k8, sq=sq, sk=sk, vin=vin, svin=svin, code=code, token=token, mode=mode):
                return _native.fp8_attn_fwd(
                    q8[:, :, :nq], k8[:, :, :nk], vin[:, :, :nk], sq[..., :nq] if token else sq,
                    sk[..., :nk] if token else sk, svin, scale_mode=code, is_causal=causal, sm_scale=sm_scale,
                    p_mode=PMODE[mode], out_dtype=BF16, return_lse=True)

            def public(causal, fn=fn, mode=mode):
                with quantum_attn.config.patch({"attention.pv_mode": mode}):
                    return fn(qc, kc, vc, is_causal=causal)
            yield Entry(f"fp8_attn_fwd {mode} {'token' if token else 'head'}", mode, run, deq(q8, sq), deq(k8, sk),
                        vc.double().cpu() if mode == "16bit" else deq(v8, sv), BF16, public)
    for dtype in (BF16, FP16):
        qd, kd, vd = (t.to(dtype).cuda() for t in (q, k, v))

        def run(nq, nk, causal, qd=qd, kd=kd, vd=vd):
            return _native.attn_fwd(qd[:, :, :nq], kd[:, :, :nk], vd[:, :, :nk], is_causal=causal, sm_scale=sm_scale,
                                    return_lse=True)

        def public(causal, qd=qd, kd=kd, vd=vd):
            return quantum_attn.attn_func(qd, kd, vd, is_causal=causal)
        yield Entry(f"attn_fwd {dtype}", "16bit", run, *(t.double().cpu() for t in (qd, kd, vd)), dtype, public)


# ------------------------------------------------------------------------------------------------ a. oracle parity
SHAPES = [
    # Sq > Skv
    (1, 2, 2, 257, 65, 64),      # the second tile is all padding
    (1, 2, 2, 1000, 300, 128),   # rows >= Skv see every key
    (1, 2, 2, 1024, 320, 256),
    (1, 2, 2, 129, 3, 128),      # Skv below one step
    (1, 2, 2, 4097, 1, 64),      # every row sees key 0 alone
    (1, 2, 2, 2100, 1030, 256),  # D 256: one-stage K / V ring, several trips
    (1, 2, 2, 1030, 333, 128),   # Skv % 4 != 0: token-wise scale_k rows are not bulk-copyable
    (2, 8, 2, 1000, 300, 128),   # batched GQA
    # Sq < Skv
    (1, 2, 2, 1, 4097, 256),     # row 0 sees key 0 alone
    (1, 2, 2, 65, 257, 64),
    (1, 2, 2, 300, 1000, 128),
    (1, 2, 2, 999, 1024, 256),
    (1, 2, 2, 128, 75600, 64),   # the tiles stop after 2 and 4 of 1 182 steps
    (2, 8, 2, 300, 1000, 64),    # batched GQA
]


@pytest.mark.parametrize("B,Hq,Hkv,Sq,Skv,D", SHAPES,
                         ids=[f"B{b}_H{hq}_{hkv}_{sq}x{skv}_d{d}" for b, hq, hkv, sq, skv, d in SHAPES])
def test_oracle_parity(B, Hq, Hkv, Sq, Skv, D):
    """O and the LSE of every entry against the fp64 oracle with the top-left mask; the public functions (one call:
    quantise + attend) give the entry's own bits."""
    q, k, v = make_inputs(B, Hq, Hkv, Sq, Skv, D, seed=Sq * 7 + Skv + D)
    for e in entries(q, k, v):
        out, lse = e.run(Sq, Skv, True)
        assert out.dtype == e.dtype
        assert torch.equal(e.public(True), out), e.tag
        p, ref_lse = probs(e.q, e.k, D**-0.5, top_left(Sq, Skv))
        check(out, lse, pv(p, e.v), ref_lse, e.mode, f"{Sq}x{Skv} d{D} {e.tag}", entry16=e.tag.startswith("attn_fwd"))


# ------------------------------------------------------------------------------------------------ b. exact structure
def assert_same_bits(a, b, tag):
    if not torch.equal(a, b):
        d = (a.float() - b.float()).abs()
        raise AssertionError(f"{tag}: {int((d != 0).sum())} of {d.numel()} differ, max {d.max().item():.3g}")


def assert_row0_is_v0(out, v_seen, mode, tag):
    """Row 0 sees key 0 alone: O = V[0].  Bit-exact where P and V stay in 16 bits; in the FP8 modes the normalisation
    1 / l multiplies the e4m3 V, so one output ulp (2^-7 relative in bf16) of the dequantised V."""
    o, ref = out[:, :, 0].double().cpu(), v_seen[:, :, 0]
    if mode == "16bit":
        assert torch.equal(o, ref), tag
    else:
        assert bool(((o - ref).abs() <= ref.abs() * 2.0**-7).all()), (tag, (o - ref).abs().max().item())


@pytest.mark.parametrize("D", [64, 128, 256])
def test_fewer_queries_is_the_square_problem_on_the_first_keys(D):
    """Sq 512 < Skv 2048: no row reaches key Sq, so the launch is, bit for bit, the square causal launch on the first Sq
    keys - same bytes, same scales.  Sq is a multiple of 256: a CTA's padding rows (which see other keys in the two
    launches and take part in the warp's rescale vote) are then absent at every D."""
    Sq, Skv = 512, 2048
    q, k, v = make_inputs(1, 2, 2, Sq, Skv, D, seed=D)
    for e in entries(q, k, v):
        out, lse = e.run(Sq, Skv, True)
        out_sq, lse_sq = e.run(Sq, Sq, True)
        assert_same_bits(out, out_sq, f"d{D} {e.tag} O")
        assert_same_bits(lse, lse_sq, f"d{D} {e.tag} LSE")
        assert_row0_is_v0(out, e.v, e.mode, f"d{D} {e.tag}")


@pytest.mark.parametrize("D", [64, 128, 256])
def test_more_queries_is_square_then_non_causal(D):
    """Sq 1536 > Skv 512: rows below Skv are, bit for bit, the square causal launch on the first Skv queries; the rows
    from Skv on see every key, masked by nothing (Skv is a multiple of 64: no ragged tail), and equal the non-causal
    launch of the same problem."""
    Sq, Skv = 1536, 512
    q, k, v = make_inputs(1, 2, 2, Sq, Skv, D, seed=D + 1)
    for e in entries(q, k, v):
        out, lse = e.run(Sq, Skv, True)
        out_sq, lse_sq = e.run(Skv, Skv, True)
        out_nc, lse_nc = e.run(Sq, Skv, False)
        assert_same_bits(out[:, :, :Skv], out_sq, f"d{D} {e.tag} O rows < Skv")
        assert_same_bits(lse[:, :, :Skv], lse_sq, f"d{D} {e.tag} LSE rows < Skv")
        assert_same_bits(out[:, :, Skv:], out_nc[:, :, Skv:], f"d{D} {e.tag} O rows >= Skv")
        assert_same_bits(lse[:, :, Skv:], lse_nc[:, :, Skv:], f"d{D} {e.tag} LSE rows >= Skv")
        assert_row0_is_v0(out, e.v, e.mode, f"d{D} {e.tag}")


@pytest.mark.parametrize("D", [64, 128, 256])
def test_one_key_gives_v0_in_every_row(D):
    """Skv = 1: every row, padding tile and all, sees key 0 alone."""
    Sq = 300
    q, k, v = make_inputs(1, 2, 2, Sq, 1, D, seed=D + 2)
    for e in entries(q, k, v):
        out, _ = e.run(Sq, 1, True)
        for r in (0, 1, 63, 64, 127, 128, 255, 256, Sq - 1):
            assert_row0_is_v0(out[:, :, r:r + 1], e.v, e.mode, f"d{D} {e.tag} row {r}")


# ------------------------------------------------------------------------------------------------ c. landscapes
@pytest.mark.parametrize("fam", ["e4m3", "16bit"])
@pytest.mark.parametrize("case", sm.RECT_CASES, ids=[c.name for c in sm.RECT_CASES])
def test_rectangular_landscape(case, fam):
    """As test_softmax_dynamics_gpu.test_landscape, on RECT_CASES: every P mode, head-wise and token-wise, and the
    16-bit entry in bf16 and fp16."""
    tau, _ = sm.tau_koff(fam == "16bit")
    design = case.make(tau)
    head = sm.landscape(design, Sq=case.Sq, Skv=case.Skv, D=case.D, seed=1)
    tok = sm.landscape(design, Sq=case.Sq, Skv=case.Skv, D=case.D, token=True, seed=1)
    ref, ref_lse = oracle_out_lse(head.x, head.dequant()[2], True)
    for mode in (("fp8", "fp8_hilo") if fam == "e4m3" else ("16bit",)):
        for L, token in ((head, False), (tok, True)):
            out, lse = run_fp8_entry(L, mode, True, token)
            check_landscape(out, lse, ref, ref_lse, mode, f"{case.name} {mode} {'token' if token else 'head'}")
    if fam == "16bit":
        for dtype in (BF16, FP16):
            out, lse = run_16bit_entry(head, dtype, True)
            check_landscape(out, lse, ref, ref_lse, "16bit", f"{case.name} attn_fwd {dtype}")


# ------------------------------------------------------------------------------------------------ d. public API
@pytest.mark.parametrize("Sq,Skv,D,dtype", [(1000, 300, 128, BF16), (300, 1000, 64, FP16), (1024, 999, 256, BF16),
                                            (999, 1024, 128, FP16)], ids=["1000x300_d128_bf16", "300x1000_d64_fp16",
                                                                          "1024x999_d256_bf16", "999x1024_d128_fp16"])
def test_public_api_against_eager_definition(Sq, Skv, D, dtype):
    """``fp8_attn_func``, ``fp8_token_wise_attn_func`` and ``attn_func`` with ``is_causal=True`` against their eager
    definition (aten quantiser + aten SDPA ``is_causal``, MATH backend: the alignment does not depend on which GPU
    backend SDPA picks).  Bounds of the public-API tests: RMSE 3e-3 with 16-bit P, the reference's 1e-2 otherwise."""
    from torch.nn.attention import SDPBackend, sdpa_kernel

    g = torch.Generator(device="cuda").manual_seed(Sq + Skv)
    q = torch.randn(1, 4, Sq, D, device="cuda", dtype=dtype, generator=g)
    k = torch.randn(1, 4, Skv, D, device="cuda", dtype=dtype, generator=g)
    v = torch.randn(1, 4, Skv, D, device="cuda", dtype=dtype, generator=g)
    rmse = lambda a, b: torch.sqrt(torch.nn.functional.mse_loss(a.float(), b.float())).item()  # noqa: E731
    with sdpa_kernel(SDPBackend.MATH):
        for fn in (quantum_attn.fp8_attn_func, quantum_attn.fp8_token_wise_attn_func):
            with quantum_attn.config.patch({"attention.force_eager_fallback": True}):
                eager = fn(q, k, v, is_causal=True)
            for mode in PMODE:
                with quantum_attn.config.patch({"attention.pv_mode": mode}):
                    out = fn(q, k, v, is_causal=True)
                assert out.dtype == dtype and out.shape == q.shape
                assert rmse(out, eager) < (3e-3 if mode == "16bit" else 1e-2), (fn.__name__, mode, rmse(out, eager))
        with quantum_attn.config.patch({"attention.force_eager_fallback": True}):
            eager = quantum_attn.attn_func(q, k, v, is_causal=True)
        assert rmse(quantum_attn.attn_func(q, k, v, is_causal=True), eager) < 3e-3


@pytest.mark.parametrize("Sq,Skv", [(1000, 300), (300, 1000)])
def test_bounds_tell_top_left_from_bottom_right(Sq, Skv):
    """The checks above would catch a kernel that aligned the mask bottom-right: its fp64 reference lies ten times or
    more outside the bounds the kernel meets against the top-left one."""
    D = 128
    q, k, v = make_inputs(1, 2, 2, Sq, Skv, D, seed=Sq + Skv)
    for e in entries(q, k, v):
        if e.mode != "16bit":
            continue
        out, lse = e.run(Sq, Skv, True)
        p, ref_lse = probs(e.q, e.k, D**-0.5, top_left(Sq, Skv))
        check(out, lse, pv(p, e.v), ref_lse, e.mode, e.tag)
        p_br, _ = probs(e.q, e.k, D**-0.5, bottom_right(Sq, Skv))
        m = oracle.compare(out.float().cpu().numpy(), pv(p_br, e.v).numpy())
        assert m["rmse_over_rms"] > 10 * REL_RMSE_BOUND[e.mode], (e.tag, m)
        assert m["max_abs_over_row_rms"] > 10 * ROW_BOUND[e.mode], (e.tag, m)
