"""The bottom-right causal mode of the C ABI (QA_CAUSAL_BOTTOM_RIGHT): row i sees keys j <= i + Skv - Sq.  The
sequence-sharded causal path attends each zig-zag chunk with it, against the keys up to the chunk's end.

The kernel takes the diagonal offset off = Skv - Sq at run time; the per-tile step counts (``nst0`` / ``nst1``), the
diagonal test, the last visible column and the first masked step (``j_mask``) all move by it.  Offsets that are not
multiples of the 64-key step or the 128-row tile put the diagonal anywhere inside a step.

* oracle parity (fp64 softmax on the inputs as the kernel reads them, O and the LSE) for every entry - ``fp8_attn_fwd``
  in the three P modes with head-wise and token-wise scales, ``attn_fwd`` in bf16 and fp16 - at D 64 / 128 / 256 and
  with batched GQA, within the bounds of tests/test_causal_rectangular_gpu.py;
* Sq == Skv: off = 0, the launch is bit for bit the top-left one;
* the rows of a bottom-right launch on the last Sq queries equal the same rows of the square top-left launch.
"""
import math

import pytest
import torch

from quantumattention_b200 import _native
from test_attention_gpu import ROW_BOUND
from test_causal_rectangular_gpu import (assert_same_bits, check, entries, make_inputs, probs, pv, row_error,
                                         top_left)
from test_softmax_dynamics_gpu import PMODE

pytestmark = pytest.mark.gpu

BR = _native.QA_CAUSAL_BOTTOM_RIGHT


def bottom_right(Sq, Skv):
    """True where a row may not look: key > row + Skv - Sq."""
    return torch.ones(Sq, Skv, dtype=torch.bool).triu(Skv - Sq + 1)


SHAPES = [(1, 2, 2, sq, skv, d) for sq, skv in ((300, 1000), (1, 777), (129, 4097), (1000, 1000)) for d in (64, 128, 256)]
SHAPES += [(2, 8, 2, 300, 1000, 128), (2, 8, 2, 129, 4097, 64)]  # batched GQA


@pytest.mark.parametrize("B,Hq,Hkv,Sq,Skv,D", SHAPES,
                         ids=[f"B{b}_H{hq}_{hkv}_{sq}x{skv}_d{d}" for b, hq, hkv, sq, skv, d in SHAPES])
def test_oracle_parity(B, Hq, Hkv, Sq, Skv, D):
    q, k, v = make_inputs(B, Hq, Hkv, Sq, Skv, D, seed=Sq * 5 + Skv + D)
    for e in entries(q, k, v):
        out, lse = e.run(Sq, Skv, BR)
        assert out.dtype == e.dtype
        p, ref_lse = probs(e.q, e.k, D**-0.5, bottom_right(Sq, Skv))
        check(out, lse, pv(p, e.v), ref_lse, e.mode, f"{Sq}x{Skv} d{D} {e.tag}", entry16=e.tag.startswith("attn_fwd"))


@pytest.mark.parametrize("S", [1000, 1024])
def test_square_is_top_left(S):
    """Sq == Skv: the offset is 0 and the launch is the top-left one, bit for bit (O and LSE)."""
    for D in (64, 128, 256):
        q, k, v = make_inputs(1, 4, 2, S, S, D, seed=S + D)
        for e in entries(q, k, v):
            out, lse = e.run(S, S, BR)
            out_tl, lse_tl = e.run(S, S, True)
            assert_same_bits(out, out_tl, f"{S} d{D} {e.tag} O")
            assert_same_bits(lse, lse_tl, f"{S} d{D} {e.tag} LSE")


@pytest.mark.parametrize("Sq,Skv,D", [(300, 1000, 128), (129, 4097, 64), (1, 777, 256), (640, 1280, 128)])
def test_rows_equal_the_square_top_left_launch(Sq, Skv, D):
    """A bottom-right launch on the LAST Sq queries is the square causal problem restricted to those rows: the same
    keys, the same visible set per row.  Same quantised bytes and head-wise scales in both launches; the rows agree
    within the row bound of each mode (bit for bit is not promised: a warp's rows share rescale decisions, and the
    warps are cut at other rows when off is not a multiple of 32)."""
    q, k, v = make_inputs(1, 4, 2, Skv, Skv, D, seed=Sq + Skv)
    qc, kc, vc = (t.to(torch.bfloat16).cuda() for t in (q, k, v))
    (q8,), (sq,) = _native.quantize_fp8([qc], _native.QA_SCALE_HEAD)
    (k8, v8), (sk, sv) = _native.quantize_fp8([kc, vc], _native.QA_SCALE_HEAD)
    off = Skv - Sq
    for mode, p_mode in PMODE.items():
        vin, svin = (vc, None) if mode == "16bit" else (v8, sv)
        kw = dict(scale_mode=_native.QA_SCALE_HEAD, sm_scale=1 / math.sqrt(D), p_mode=p_mode, out_dtype=torch.bfloat16)
        full = _native.fp8_attn_fwd(q8, k8, vin, sq, sk, svin, is_causal=True, **kw)
        part = _native.fp8_attn_fwd(q8[:, :, off:], k8, vin, sq, sk, svin, is_causal=BR, **kw)
        ref = full[:, :, off:].double().cpu()
        assert row_error(part, ref) <= ROW_BOUND[mode], (mode, row_error(part, ref))
        if off % 128 == 0:  # tiles cut at the same rows: identical
            assert_same_bits(part, full[:, :, off:], f"{Sq}x{Skv} {mode}")
    for dtype in (torch.bfloat16, torch.float16):
        qd, kd, vd = (t.to(dtype).cuda() for t in (q, k, v))
        full = _native.attn_fwd(qd, kd, vd, is_causal=True, sm_scale=1 / math.sqrt(D))
        part = _native.attn_fwd(qd[:, :, off:], kd, vd, is_causal=BR, sm_scale=1 / math.sqrt(D))
        assert row_error(part, full[:, :, off:].double().cpu()) <= ROW_BOUND["16bit"], dtype


def test_mask_differs_from_top_left():
    """The parity checks tell the two alignments apart: a bottom-right launch is far outside the bounds against the
    top-left reference of the same rectangular problem."""
    Sq, Skv, D = 300, 1000, 128
    q, k, v = make_inputs(1, 2, 2, Sq, Skv, D, seed=3)
    for e in entries(q, k, v):
        if e.mode != "16bit":
            continue
        out, _ = e.run(Sq, Skv, BR)
        p_tl, _ = probs(e.q, e.k, D**-0.5, top_left(Sq, Skv))
        assert row_error(out, pv(p_tl, e.v)) > 10 * ROW_BOUND["16bit"], e.tag
