"""The designed softmax landscapes (oracle/softmax_model.py) do what tests/test_softmax_dynamics_gpu.py relies on:
their bytes decode to exactly the designed scores, and the kernel's lazy-rescale rule, replayed on them, rescales at
the intended steps and keeps p' inside the headroom of the P type.  Without these checks the GPU tests could quietly
turn back into tests of random inputs, which almost never reach the rescale path."""
import math

import numpy as np
import pytest

import oracle
from oracle import softmax_model as sm


@pytest.mark.parametrize("level", [4.25, 68.25, 4 + 2.0**-6, -131.5, 60.0, 57.75, 3 + 5 / 64, 0.0])
def test_levels_decompose_exactly(level):
    parts = sm.decompose(level)
    assert len(parts) == 3 and sum(parts) == level
    assert np.array_equal(oracle.e4m3_decode(oracle.e4m3_encode_rne_sat(np.float32(parts))), np.float32(parts))


def test_level_that_is_no_e4m3_sum_is_refused():
    with pytest.raises(ValueError):
        sm.decompose(1 + 2.0**-12)  # below the smallest e4m3 subnormal, 2^-9


def _check_bytes(L, token):
    for b in (L.q8, L.k8, L.v8):
        assert not np.isin(b, (0x7F, 0xFF)).any()  # no NaN bytes
    q, k, v = L.dequant()
    rep = q.shape[1] // k.shape[1]
    assert np.array_equal(np.matmul(q, np.repeat(k, rep, axis=1).swapaxes(-1, -2)), L.x)
    assert np.array_equal(v.astype(np.float32).astype(np.float64), v)
    if token:  # every token carries a power of two, and not all of them are 1
        for s in (L.scale_q, L.scale_k):
            e = np.log2(s)
            assert np.array_equal(e, np.round(e)) and e.min() >= -3 and e.max() <= 3 and (e != 0).mean() > 0.5


@pytest.mark.parametrize("fam", ["16bit", "e4m3"])
@pytest.mark.parametrize("case", sm.CASES + sm.RECT_CASES, ids=[c.name for c in sm.CASES + sm.RECT_CASES])
def test_landscape_drives_the_intended_rescales(case, fam):
    tau, koff = sm.tau_koff(fam == "16bit")
    design = case.make(tau)
    head = sm.landscape(design, Sq=case.Sq, Skv=case.Skv, D=case.D, seed=1)
    tok = sm.landscape(design, Sq=case.Sq, Skv=case.Skv, D=case.D, token=True, seed=1)
    _check_bytes(head, False)
    _check_bytes(tok, True)
    assert np.array_equal(head.x, tok.x) and np.array_equal(head.v8, tok.v8)
    r = sm.rescale_events(head.x, v16=fam == "16bit", causal=case.causal, D=case.D)
    assert sorted({j for (_, _, _, j) in r.events}) == list(case.expect), (case.name, fam)
    if design.rows == "tile1":
        assert all((w * sm.WARP // sm.BM) % 2 == 1 for (_, _, w, _) in r.events)
    assert r.max_exp <= koff + tau - 2 * sm.ETA + 1e-12  # headroom, with the noise margin
    if fam == "e4m3":
        assert 2.0**r.max_exp <= sm.E4M3_P_HEADROOM <= sm.E4M3_P_MAX
    if "below" in case.name:  # the headroom cases come within 1/4 + 2 ETA of it
        assert r.max_exp >= koff + tau - 0.25 - 2 * sm.ETA


@pytest.mark.parametrize("fam", ["16bit", "e4m3"])
@pytest.mark.parametrize("case", sm.RECT_CASES, ids=[c.name for c in sm.RECT_CASES])
def test_rectangular_landscape_rescales_the_intended_warps(case, fam):
    """Causal with Sq != Skv: only the warps whose rows reach the raised keys rescale, and keys past every row's
    diagonal leave the masked LSE alone while they would dominate it unmasked."""
    tau, _ = sm.tau_koff(fam == "16bit")
    L = sm.landscape(case.make(tau), Sq=case.Sq, Skv=case.Skv, D=case.D, seed=1)
    r = sm.rescale_events(L.x, v16=fam == "16bit", causal=True, D=case.D)
    assert {w for (_, _, w, _) in r.events} == set(sm.RECT_WARPS.get(case.name, ())), case.name
    if case.Sq < case.Skv:
        assert sm.logsumexp_ref(L.x, causal=True).max() < math.log(case.Sq) + sm.ETA  # Sq keys of level ~0 at most
        assert sm.logsumexp_ref(L.x, causal=False).min() > 59 * sm.LN2


def test_long_landscape_drives_the_intended_rescales():
    case = sm.LONG
    for fam in ("16bit", "e4m3"):
        tau, koff = sm.tau_koff(fam == "16bit")
        L = sm.landscape(case.make(tau), Sq=case.Sq, Skv=case.Skv, D=case.D, seed=1)
        assert -(-case.Skv // sm.BS) == 1182 and case.Skv - 1181 * sm.BS == 16
        q, k, _ = L.dequant()
        assert np.array_equal(np.matmul(q, k.swapaxes(-1, -2)), L.x)
        r = sm.rescale_events(L.x, v16=fam == "16bit", causal=False, D=case.D)
        assert sorted({j for (_, _, _, j) in r.events}) == list(case.expect)
        assert r.max_exp <= koff + tau


def test_random_inputs_barely_reach_the_rescale_path():
    """Why the landscapes exist: randn scores move a 16-bit-P row maximum by more than TAU in no step."""
    q, k, _ = oracle.make_qkv(1, 2, 1024, 1024, 128, seed=1024 + 128)
    (q8, sq), (k8, sk) = oracle.quantize_fp8(q.float().numpy()), oracle.quantize_fp8(k.float().numpy())
    qh, kh = oracle.dequantize(q8, sq).astype(np.float64), oracle.dequantize(k8, sk).astype(np.float64)
    x = (qh @ kh.swapaxes(-1, -2)) / math.sqrt(128) / math.log(2)
    assert not sm.rescale_events(x, v16=True, causal=False, D=128).events


def test_rule_replay_on_a_hand_made_row():
    """The replay against a case worked by hand: one warp, steps 0-3 at levels 0, 5, 9, 9.5 (e4m3 P: TAU = 4)."""
    x = np.zeros((1, 1, 32, 256))
    for j, lv in enumerate((0.0, 5.0, 9.0, 9.5)):
        x[..., j * 64:(j + 1) * 64] = lv
    x[0, 0, 1:] = 0.0  # one row of the warp moves, the other 31 stay flat
    r = sm.rescale_events(x, v16=False, causal=False, D=256, qtmem=False)
    # step 1: 5 > 4 -> rescale (m_used = 5); step 2: 4 -> no; step 3: 4.5 > 4 -> rescale; p' tops out at 2^(4 + 4)
    assert r.events == {(0, 0, 0, 1), (0, 0, 0, 3)}
    assert r.max_exp == 8.0
