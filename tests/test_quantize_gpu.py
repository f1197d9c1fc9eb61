"""Parity of the sm_100a quantiser with the oracle: BIT-EXACT bytes and scales (integer / byte work)."""
import os
import zlib

import numpy as np
import pytest
import torch

import oracle
import quantum_attn
from quantumattention_b200 import _native
from conftest import bf16_from_bits

pytestmark = pytest.mark.gpu

# "head-wise-2pass": same function through the two-pass kernels (what heads longer than one resident wave take)
MODES = {"head-wise": _native.QA_SCALE_HEAD, "token-wise": _native.QA_SCALE_TOKEN,
         "head-wise-2pass": _native.QA_SCALE_HEAD_TWO_PASS}


def _check(x_cpu: torch.Tensor, mode: str):
    (x8,), (scale,) = _native.quantize_fp8([x_cpu.cuda()], MODES[mode])
    torch.cuda.synchronize()
    b, s = oracle.quantize_fp8(x_cpu.float().numpy(), mode.replace("-2pass", ""))
    got = x8.view(torch.uint8).cpu().numpy()
    assert got.shape == b.shape
    nbad = int((got != b).sum())
    assert nbad == 0, f"{nbad} of {b.size} bytes differ"
    assert np.array_equal(scale.cpu().numpy(), s)


@pytest.mark.parametrize("mode,file", [("head-wise", "quantize_head.npz"), ("token-wise", "quantize_token.npz")])
def test_golden_vectors_from_reference(golden_dir, mode, file):
    g = np.load(os.path.join(golden_dir, file))
    x = bf16_from_bits(g["x_bf16_bits"])
    (x8,), (scale,) = _native.quantize_fp8([x.cuda()], MODES[mode])
    assert np.array_equal(x8.view(torch.uint8).cpu().numpy(), g["q_bytes"])
    assert np.array_equal(scale.cpu().numpy(), g["scale"])


@pytest.mark.parametrize("mode", ["head-wise", "token-wise", "head-wise-2pass"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", [(2, 8, 512, 64), (1, 3, 999, 128), (1, 2, 1000, 256), (1, 1, 1, 64), (2, 2, 17, 128)])
def test_random_inputs(mode, dtype, shape):
    # (zlib.crc32, not hash(): str hashes are salted per process and the test must draw the same tensors every run)
    g = torch.Generator().manual_seed(zlib.crc32(repr((mode, str(dtype), shape)).encode()))
    x = (torch.randn(shape, generator=g) * torch.exp(torch.randn(shape[:2] + (1, shape[3]), generator=g))).to(dtype)
    _check(x, mode)


@pytest.mark.parametrize("mode", ["head-wise", "token-wise", "head-wise-2pass"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_signed_zeros_and_underflow(mode, dtype):
    # -0.0 inputs (a 16-bit underflow of a small negative number) must encode as 0x80 like the reference's division
    g = torch.Generator().manual_seed(77)
    x = torch.randn((1, 2, 200, 128), generator=g)
    x[0, 0, ::3, ::5] = -0.0
    x[0, 1, 1::7, 3::11] = 0.0
    x[0, 1, 5, :] = -1e-7   # flushes to -0 in fp16, stays a tiny normal in bf16
    x[0, 0, 9, :] = torch.tensor(-6e-8)  # fp16 subnormal
    _check(x.to(dtype), mode)


@pytest.mark.parametrize("kind", ["outlier_channels", "huge_token", "zero_head"])
@pytest.mark.parametrize("mode", ["head-wise", "token-wise", "head-wise-2pass"])
def test_stress_inputs(kind, mode):
    q, k, v = oracle.make_qkv(1, 3, 300, 300, 128, seed=5, kind=kind)
    for t in (q, k, v):
        _check(t, mode)


def test_three_tensors_one_launch_and_ragged_lengths():
    q, k, v = oracle.make_qkv(2, 4, 333, 470, 128, seed=9)
    (q8, k8, v8), (sq, sk, sv) = _native.quantize_fp8([q.cuda(), k.cuda(), v.cuda()], _native.QA_SCALE_HEAD)
    assert _native.last_launch_count() == 1  # single-pass head-wise kernel, Q, K and V in one launch
    for t, t8, s in ((q, q8, sq), (k, k8, sk), (v, v8, sv)):
        b, sc = oracle.quantize_fp8(t.float().numpy(), "head-wise")
        assert np.array_equal(t8.view(torch.uint8).cpu().numpy(), b)
        assert np.array_equal(s.cpu().numpy(), sc)


def test_strided_input_views():
    base = torch.randn(2, 300, 4, 128, generator=torch.Generator().manual_seed(2)).to(torch.bfloat16)
    x = base.permute(0, 2, 1, 3)  # [B,H,S,D] view of a [B,S,H,D] buffer, as DiT code often holds it
    assert not x.is_contiguous()
    (x8,), (scale,) = _native.quantize_fp8([x.cuda()], _native.QA_SCALE_HEAD)
    b, s = oracle.quantize_fp8(x.float().numpy(), "head-wise")
    assert np.array_equal(x8.view(torch.uint8).cpu().numpy(), b) and np.array_equal(scale.cpu().numpy(), s)


def test_public_dynamically_quantize_fp8():
    # reference signature: dynamically_quantize_fp8(t, *, reduction_dim=-1) -> (t_fp8, scale) (nn.py:22-42)
    x = torch.randn(2, 4, 100, 64, generator=torch.Generator().manual_seed(1)).to(torch.float16)
    t8, s = quantum_attn.dynamically_quantize_fp8(x.cuda())
    b, sc = oracle.quantize_fp8(x.float().numpy(), "token-wise")
    assert t8.dtype == torch.float8_e4m3fn and s.shape == (2, 4, 100) and s.dtype == torch.float32
    assert np.array_equal(t8.view(torch.uint8).cpu().numpy(), b) and np.array_equal(s.cpu().numpy(), sc)
    t8, s = quantum_attn.dynamically_quantize_fp8(x.cuda(), reduction_dim=[2, 3])
    b, sc = oracle.quantize_fp8(x.float().numpy(), "head-wise")
    assert s.shape == (2, 4)
    assert np.array_equal(t8.view(torch.uint8).cpu().numpy(), b) and np.array_equal(s.cpu().numpy(), sc)
    with pytest.raises(ValueError):
        quantum_attn.dynamically_quantize_fp8(x.cuda(), reduction_dim=0)


def test_full_size_checksum_flux_shape():
    # BASELINE config C2 (FLUX): too big for the numpy oracle in seconds -> size-independent properties instead:
    # (1) decode(encode(x)) is within half an e4m3 step of x / scale, (2) idempotence: re-quantising the dequantised
    # tensor reproduces the same bytes, (3) scale == amax/448 exactly.
    q, _, _ = oracle.make_qkv(1, 24, 4608, 4608, 128, seed=0)
    x = q.cuda()
    (x8,), (scale,) = _native.quantize_fp8([x], _native.QA_SCALE_HEAD)
    amax = x.float().abs().amax(dim=(2, 3))
    assert torch.equal(scale, (amax * (1.0 / 448.0)).clamp_min(torch.finfo(torch.float32).eps))
    deq = x8.float() * scale[:, :, None, None]
    y = x.float() / scale[:, :, None, None]
    err = (x8.float() - y).abs()
    step = torch.where(y.abs() < 2.0**-6, torch.tensor(2.0**-9, device="cuda"),
                       torch.exp2(torch.floor(torch.log2(y.abs().clamp_min(2.0**-6))) - 3))
    assert bool((err <= 0.5 * step * 1.0001).all())
    (x8b,), (scale_b,) = _native.quantize_fp8([deq.to(torch.bfloat16)], _native.QA_SCALE_HEAD)
    # bf16 rounding of deq may move a value across an e4m3 rounding boundary only if it was not representable;
    # e4m3 * power-of-two-ish scale is exactly representable in bf16 only when scale has <= 5 mantissa bits, so
    # compare on the fp32 path instead: quantise(deq) in torch with the same formula
    y2 = (deq / scale[:, :, None, None]).clamp(-448, 448).to(torch.float8_e4m3fn)
    assert torch.equal(y2.view(torch.uint8), x8.view(torch.uint8))


def test_single_pass_matches_two_pass_at_flux_size():
    """C2-sized tensors (36 CTAs per head, 2592 CTAs): the per-head arrival protocol against the two-pass kernels."""
    q, k, v = oracle.make_qkv(1, 24, 4608, 4608, 128, seed=3)
    xs = [q.cuda(), k.cuda(), v.cuda()]
    for _ in range(3):  # repeated calls: the workspace is re-zeroed per call
        a8, asc = _native.quantize_fp8(xs, _native.QA_SCALE_HEAD)
    assert _native.last_launch_count() == 1
    b8, bsc = _native.quantize_fp8(xs, _native.QA_SCALE_HEAD_TWO_PASS)
    assert _native.last_launch_count() == 2
    for x8, y8, s1, s2 in zip(a8, b8, asc, bsc):
        assert torch.equal(x8.view(torch.uint8), y8.view(torch.uint8))
        assert torch.equal(s1, s2)
    b, sc = oracle.quantize_fp8(q[:, :2].float().numpy(), "head-wise")
    assert np.array_equal(a8[0][:, :2].view(torch.uint8).cpu().numpy(), b)
    assert np.array_equal(asc[0][:, :2].cpu().numpy(), sc)


def test_long_head_takes_two_pass_path():
    """A head of 150k tokens at D=64 exceeds one resident wave even with 16 passes per CTA -> two launches."""
    g = torch.Generator().manual_seed(11)
    x = torch.randn(1, 1, 400_000, 64, generator=g).to(torch.bfloat16)
    (x8,), (scale,) = _native.quantize_fp8([x.cuda()], _native.QA_SCALE_HEAD)
    n = _native.last_launch_count()
    b, sc = oracle.quantize_fp8(x.float().numpy(), "head-wise")
    assert np.array_equal(x8.view(torch.uint8).cpu().numpy(), b) and np.array_equal(scale.cpu().numpy(), sc)
    assert n in (1, 2)


@pytest.mark.parametrize("shape,n_tensors", [((1, 2, 75600, 128), 3), ((1, 1, 60000, 256), 1), ((2, 1, 100001, 64), 2)])
def test_long_heads_reload_mode_is_head_wise(shape, n_tensors):
    """Heads that span 4 - 10 trips of the grid (the long-video shape: 591 slabs per head on 148 SMs), through the
    default head-wise mode and through QA_SCALE_HEAD_RELOAD, which ABI 6 callers may still pass: both take the same
    kernels, and their bytes and scales are identical to the oracle and to the two-pass kernels, ragged lengths and
    several tensors included."""
    g = torch.Generator().manual_seed(shape[2])
    xs = [(torch.randn(shape, generator=g) * (1.0 + i)).to(torch.bfloat16) for i in range(n_tensors)]
    if n_tensors > 1:  # ragged: a shorter second tensor
        xs[1] = xs[1][:, :, : shape[2] - 777].contiguous()
    xc = [x.cuda() for x in xs]
    outs, scales = _native.quantize_fp8(xc, _native.QA_SCALE_HEAD_RELOAD)
    n_reload = _native.last_launch_count()
    outs1, scales1 = _native.quantize_fp8(xc, _native.QA_SCALE_HEAD)
    assert _native.last_launch_count() == n_reload
    outs2, scales2 = _native.quantize_fp8(xc, _native.QA_SCALE_HEAD_TWO_PASS)
    for x, o, sc, o1, sc1, o2, sc2 in zip(xs, outs, scales, outs1, scales1, outs2, scales2):
        assert torch.equal(o.view(torch.uint8), o2.view(torch.uint8)) and torch.equal(sc, sc2)
        assert torch.equal(o1.view(torch.uint8), o2.view(torch.uint8)) and torch.equal(sc1, sc2)
        b, s_ = oracle.quantize_fp8(x.float().numpy(), "head-wise")
        assert np.array_equal(sc.cpu().numpy(), s_) and np.array_equal(o.view(torch.uint8).cpu().numpy(), b)
    # back to back on the persistent workspace, other shapes in between
    _native.quantize_fp8([xc[0][:, :, :5000].contiguous()], _native.QA_SCALE_HEAD)
    outs3, scales3 = _native.quantize_fp8(xc, _native.QA_SCALE_HEAD_RELOAD)
    for o, o3, sc, sc3 in zip(outs, outs3, scales, scales3):
        assert torch.equal(o.view(torch.uint8), o3.view(torch.uint8)) and torch.equal(sc, sc3)


def test_quotient_is_correctly_rounded_for_adversarial_scales():
    """The reciprocal-plus-correction quotient must give the bytes of IEEE division: bytes identical to the oracle for scales
    whose mantissa is all ones / just above a power of two (worst cases for reciprocal rounding), and every bf16
    magnitude below amax as the numerator."""
    bits = torch.arange(0, 0x7F80, dtype=torch.int32).to(torch.int16)  # every non-negative finite bf16
    allv = bits.view(torch.bfloat16).float()
    for amax in (448.0 * 1.99999988, 448.0 * 1.00000012, 3.0, 0.333251953125, 1.0e-3, 57344.0, 1.00390625):
        amax_bf = torch.tensor(amax).to(torch.bfloat16).float().item()
        vals = allv[allv <= amax_bf]
        n = (vals.numel() // 64) * 64
        x = vals[-n:].clone()
        x[-1] = amax_bf
        x = torch.cat([x, -x]).reshape(1, 1, -1, 64).to(torch.bfloat16)
        _check(x, "head-wise")
        _check(x, "token-wise")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_every_numerator_under_sampled_amax(dtype):
    """The quantiser divides by its own scale with a reciprocal and ONE residual correction; that this yields the
    reference's byte was decided by enumerating all (amax, x) pairs on the CPU (scripts/ubench/div_exhaustive.c).  Here
    the kernels themselves see every 16-bit magnitude (both signs) under each of 96 sampled amax values per dtype -
    subnormal, tiny (scale clamped to eps), mid-range and largest-finite included."""
    top = 0x7F7F if dtype == torch.bfloat16 else 0x7BFF
    rng = np.random.default_rng(20260 + top)
    amax_bits = np.unique(np.concatenate([[1, 2, 0x7F, 0x80, 0x81, 0x3F80, 0x3C00, 0x0400, 0x03FF, top - 1, top],
                                          rng.integers(1, top + 1, size=120)]))[:96]
    mags = np.arange(0, 0x8000, dtype=np.int64)
    heads = []
    for ab in amax_bits:
        m = np.where(mags <= ab, mags, 0)          # magnitudes order like their bit patterns
        m[0] = ab
        heads.append(np.concatenate([m, m | 0x8000]).astype(np.uint16))
    bits = np.stack(heads).reshape(1, len(heads), 512, 128).view(np.int16)
    x = torch.from_numpy(bits.copy()).view(dtype)
    for mode in ("head-wise", "head-wise-2pass", "token-wise"):
        _check(x, mode)


def test_persistent_workspace_across_shapes_and_paths():
    """QA_WS_PERSISTENT (include/qattn.h): one zeroed-once workspace serves calls of different shapes through the
    single-pass and the two-pass kernels in any order - slots are matched by generation tag, never by stale bytes."""
    shapes = [(1, 6, 4608, 128), (2, 8, 512, 64), (1, 2, 1000, 256), (1, 24, 300, 128), (2, 8, 512, 64), (1, 3, 999, 128)]
    for i, shape in enumerate(shapes * 2):
        g = torch.Generator().manual_seed(100 + i)
        x = torch.randn(shape, generator=g).to(torch.bfloat16)
        _check(x, "head-wise-2pass" if i % 3 == 1 else "head-wise")


def test_plain_scratch_workspace_full_of_garbage():
    """Without the flag the workspace is plain scratch: whatever it holds (here words that look like valid tags) is
    cleared by the call."""
    x = torch.randn((1, 4, 2048, 128), generator=torch.Generator().manual_seed(3)).to(torch.bfloat16)
    n = int(_native.load().qa_quantize_workspace_floats(1, 4, 2048, 128))
    for fill in (-1, 1, 2, 3, 7, 1000):
        ws = torch.full((n,), fill, dtype=torch.int32, device="cuda").view(torch.float32)
        (x8,), (scale,) = _native.quantize_fp8([x.cuda()], _native.QA_SCALE_HEAD, workspace=ws)
        b, s = oracle.quantize_fp8(x.float().numpy(), "head-wise")
        assert np.array_equal(x8.view(torch.uint8).cpu().numpy(), b) and np.array_equal(scale.cpu().numpy(), s)


def test_two_streams_quantise_concurrently_without_deadlock():
    """The single-pass kernel's CTAs wait for each other (one CTA per SM): two such grids on different streams must
    not split the SMs between them and spin forever.  They are launched cooperatively - a grid is scheduled only once
    it fits as a whole - so concurrent calls queue; results stay byte-exact.  (Each stream has its own workspace.)"""
    g = torch.Generator().manual_seed(21)
    xs = [torch.randn(1, 24, 4608, 128, generator=g).to(torch.bfloat16).cuda() for _ in range(2)]
    refs = [oracle.quantize_fp8(x.float().cpu().numpy(), "head-wise") for x in xs]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    torch.cuda.synchronize()
    outs = [None, None]
    for rep in range(25):
        for i, st in enumerate(streams):
            with torch.cuda.stream(st):
                outs[i] = _native.quantize_fp8([xs[i]], _native.QA_SCALE_HEAD)
    torch.cuda.synchronize()
    for i in range(2):
        (x8,), (sc,) = outs[i]
        assert np.array_equal(sc.cpu().numpy(), refs[i][1]) and np.array_equal(x8.view(torch.uint8).cpu().numpy(), refs[i][0])
