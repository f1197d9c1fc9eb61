"""Designed score landscapes for the fused kernel's online softmax, and a model of its lazy-rescale rule (TEST
INFRASTRUCTURE ONLY).

Random inputs almost never move a row maximum by more than TAU within one 64-key step, so they leave the kernel's
rescale path (``attn_fwd_kernel.cuh``: the warp vote on ``(max(S_{j+1}) - m_used) * c > TAU`` and the rescale of O
and L behind it) unexercised.  ``landscape`` builds inputs whose scores, in the kernel's base-2 domain, are chosen
dyadic values, so a test can put a rescale (or its absence) at a chosen step, warp and query tile:

* scale 1 and ``sm_scale = ln 2`` make the base-2 multiplier c = 1 (up to fp32 rounding of ln 2 * log2 e);
* three "level" channels (q = 1 on every row) carry a per-key level, split greedily into at most three e4m3 values
  whose sum is exact;
* three "selector" channels carry a per-key level that only the selected rows see (q = 1 there, 0 elsewhere);
* one noise channel, |q| <= 1/4 and |k| <= 1/4, adds at most ETA = 1/16 to a score;
* every other channel is zero, and V is ``randn`` rounded to e4m3 with a power-of-two scale, so the same values are
  exact as e4m3, bf16 and fp16 and one fp64 oracle serves every entry point.

Token-wise variants put per-token powers of two on ``scale_q`` / ``scale_k`` and divide them out of the bytes: the
dequantised scores stay the same, so the kernel's vote has to see the scaled scores.

``rescale_events`` replays the rule on the designed scores.  Tests use it to prove that a landscape drives the
intended rescales, never to produce the expected output.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

from .e4m3 import decode_table, e4m3_decode, e4m3_encode_rne_sat

BS = 64     # keys per softmax step (attn_fwd_kernel.cuh: BS)
BM = 128    # query rows per tile (BM)
WARP = 32   # rows per vote
ETA = 1.0 / 16  # largest |noise| added to a score
E4M3_P_MAX = 448.0
LN2 = math.log(2.0)

CH_LEVEL = (0, 1, 2)
CH_SEL = (3, 4, 5)
CH_NOISE = 6


def tau_koff(v16: bool):
    """(TAU, KOFF) of the kernel: mirrors AttnCfg::TAU / AttnCfg::KOFF (attn_fwd_kernel.cuh:131-133).  p' =
    2^KOFF * exp2(s - m_used), and m_used may lag the true row maximum by up to TAU (log2 units) before a rescale."""
    return (8.0, 0.0) if v16 else (4.0, 4.0)


def n_tiles_per_cta(D: int) -> int:
    """Query tiles per CTA (AttnCfg::NQ): two for D <= 128, one at D = 256."""
    return 2 if D <= 128 else 1


# ------------------------------------------------------------------------------------------------ e4m3 sums
_POS = np.unique(decode_table()[:0x7F].astype(np.float64))  # non-negative finite e4m3 values, ascending


def decompose(level: float, parts: int = 3):
    """``level`` as a sum of at most ``parts`` e4m3 values (greedy: the largest one not above what is left).
    Raises if the sum cannot be exact."""
    out, rest = [], abs(float(level))
    sign = -1.0 if level < 0 else 1.0
    while rest > 0 and len(out) < parts:
        v = _POS[np.searchsorted(_POS, rest, side="right") - 1]
        out.append(sign * v)
        rest -= v
    if rest != 0:
        raise ValueError(f"level {level} is not a sum of {parts} e4m3 values")
    return out + [0.0] * (parts - len(out))


# ------------------------------------------------------------------------------------------------ designs
@dataclass(frozen=True)
class Design:
    """Per-key levels in log2 units: ``level`` is seen by every row, ``sel_level`` by the rows ``rows`` selects
    ("all", "lane17" = row 17 of every warp, "tile1" = the second 128-row tile of every 256 rows).  ``quiet`` keys
    carry no noise."""
    name: str
    level: tuple = ()       # ((first_key, value), ...): piecewise constant, 0 before the first entry
    sel_level: tuple = ()
    rows: str = "all"
    quiet: tuple = ()
    point: tuple = ()       # ((key, value), ...): single keys of `level` (applied after the pieces)
    floor: float = 0.0      # level of every key not otherwise set when `point` is used

    def key_levels(self, Skv: int):
        lv = np.full(Skv, self.floor if self.point else 0.0)
        for first, val in self.level:
            lv[first:] = val
        for key, val in self.point:
            if key < Skv:
                lv[key] = val
        sl = np.zeros(Skv)
        for first, val in self.sel_level:
            sl[first:] = val
        return lv, sl

    def row_mask(self, Sq: int):
        r = np.arange(Sq)
        if self.rows == "all":
            return np.ones(Sq, bool)
        if self.rows == "lane17":
            return r % WARP == 17
        if self.rows == "tile1":
            return (r // BM) % 2 == 1
        raise ValueError(self.rows)


def jump(J: int, delta: float, rows: str = "all") -> Design:
    """The selected rows' scores rise by ``delta`` at the first key of step J and stay there."""
    return Design(f"jump(J={J},d={delta},{rows})", sel_level=((J * BS, delta),), rows=rows)


def staircase(delta: float, first: int, last: int, rows: str = "all") -> Design:
    """The scores rise by ``delta`` at the start of every step first+1 .. last and stay at the top afterwards."""
    return Design(f"stairs(d={delta},{first}..{last},{rows})",
                  sel_level=tuple(((j * BS), (j - first) * delta) for j in range(first + 1, last + 1)), rows=rows)


def descending(drop: float = 130.0) -> Design:
    """Key 0 at level 0, every later key ``drop`` below it: p' of those keys lies under the polynomial's -125 clamp,
    under MUFU.EX2's flush to zero and under fp16's smallest subnormal."""
    return Design(f"descending({drop})", level=((1, -drop),))


def spike(J: int, delta: float, floor: float = -24.0) -> Design:
    """A noise-free key 0 at level 0 and one noise-free key in step J at ``delta`` (0 < delta <= TAU: no vote), every
    other key at ``floor``.  The spike dominates its row, and p' = 2^(KOFF + delta) is rounded to e4m3 with a relative
    error close to the largest possible - the case that bounds the single-e4m3 LSE."""
    k = J * BS + 5
    return Design(f"spike(J={J},d={delta})", point=((0, 0.0), (k, delta)), floor=floor, quiet=(0, k))


# ------------------------------------------------------------------------------------------------ inputs
@dataclass
class Landscape:
    x: np.ndarray        # fp64 [B,H,Sq,Skv]: designed scores in log2 units (before any mask)
    q8: np.ndarray       # uint8 e4m3 [B,H,Sq,D]
    k8: np.ndarray       # uint8 e4m3 [B,Hkv,Skv,D]
    scale_q: np.ndarray  # fp32 [B,H] (head-wise) or [B,H,Sq] (token-wise)
    scale_k: np.ndarray
    v8: np.ndarray       # uint8 e4m3 [B,Hkv,Skv,D]
    scale_v: np.ndarray  # fp32 [B,Hkv], powers of two
    sm_scale: float = LN2

    def dequant(self):
        """fp64 Q, K, V as the kernel sees them (exact in bf16 and fp16 as well)."""
        def dq(b, s):
            v = e4m3_decode(b).astype(np.float64)
            s = np.asarray(s, np.float64)
            while s.ndim < v.ndim:
                s = s[..., None]
            return v * s
        return dq(self.q8, self.scale_q), dq(self.k8, self.scale_k), dq(self.v8, self.scale_v)


def _exact_pow2_exponents(vals: np.ndarray, rng, lo=-3, hi=3):
    """Per row of ``vals`` (tokens x channels, e4m3 values): a random e in [lo, hi] such that every value / 2^e is
    still an exact e4m3 value."""
    es = np.arange(lo, hi + 1)
    ok = np.stack([(e4m3_decode(e4m3_encode_rne_sat((vals / 2.0**e).astype(np.float32))) == vals / 2.0**e).all(-1)
                   for e in es], -1)  # [tokens, exponents]; e = 0 is always exact
    pick = rng.random(ok.shape) * ok
    return es[pick.argmax(-1)]


def landscape(design: Design, *, B=1, H=2, Hkv=None, Sq, Skv, D, token=False, seed=0) -> Landscape:
    Hkv = H if Hkv is None else Hkv
    rng = np.random.default_rng(seed)
    lv, sl = design.key_levels(Skv)
    rows = design.row_mask(Sq)
    k = np.zeros((B, Hkv, Skv, D))
    q = np.zeros((B, H, Sq, D))
    cache = {}  # (levels are piecewise constant: each distinct value is decomposed once)

    def parts(v):
        if v not in cache:
            cache[v] = decompose(v)
        return cache[v]

    k[..., list(CH_LEVEL)] = np.array([parts(v) for v in lv])
    k[..., list(CH_SEL)] = np.array([parts(v) for v in sl])
    q[..., list(CH_LEVEL)] = 1.0
    q[..., list(CH_SEL)] = rows[:, None].astype(np.float64)
    # noise: multiples of 2^-6 in [-1/4, 1/4] on both sides, so every product is exact and at most 1/16
    qn = rng.integers(-16, 17, size=(B, H, Sq)) / 64.0
    kn = rng.integers(-16, 17, size=(B, Hkv, Skv)) / 64.0
    kn[..., list(design.quiet)] = 0.0
    q[..., CH_NOISE] = qn
    k[..., CH_NOISE] = kn
    vr = rng.standard_normal((B, Hkv, Skv, D))  # (drawn before the token scales: the same V in both variants)
    x = np.matmul(q, np.repeat(k, H // Hkv, axis=1).swapaxes(-1, -2))

    if token:
        eq = _exact_pow2_exponents(q.reshape(-1, D), rng).reshape(B, H, Sq)
        ek = _exact_pow2_exponents(k.reshape(-1, D), rng).reshape(B, Hkv, Skv)
        scale_q, scale_k = np.exp2(eq).astype(np.float32), np.exp2(ek).astype(np.float32)
        q, k = q / scale_q[..., None], k / scale_k[..., None]
    else:
        scale_q, scale_k = np.ones((B, H), np.float32), np.ones((B, Hkv), np.float32)
    q8 = e4m3_encode_rne_sat(q.astype(np.float32))
    k8 = e4m3_encode_rne_sat(k.astype(np.float32))
    v8 = e4m3_encode_rne_sat((vr * 64.0).astype(np.float32))
    return Landscape(x=x, q8=q8, k8=k8, scale_q=scale_q, scale_k=scale_k, v8=v8,
                     scale_v=np.full((B, Hkv), 1.0 / 64.0, np.float32))


# ------------------------------------------------------------------------------------------------ the rule
@dataclass
class Replay:
    events: set          # {(b, h, warp, j)}: warp = global query row // 32, j >= 1 the step that rescales
    max_exp: float       # largest p' exponent, log2 units: KOFF + s - m_used
    steps: int           # 64-key steps of the last query tile (causal: of the diagonal's tile)


def rescale_events(x: np.ndarray, *, v16: bool, causal: bool, D: int, qtmem: bool = None) -> Replay:
    """Replay the kernel's lazy-rescale rule on scores ``x`` [B,H,Sq,Skv] (log2 units).

    Per warp of 32 rows: step 0 sets m_used to the row maximum of S_0; in step j >= 1 the warp rescales if some row's
    maximum of S_j exceeds its m_used by more than TAU, and then every row of the warp takes max(m_used, max S_j).
    Rows past Sq are modelled as the kernel computes them: copies of row Sq - 1 where Q is loaded into tensor memory
    (``qtmem``: e4m3 Q/K at D = 256), zero scores where the TMA fills them with zeros.
    """
    tau, koff = tau_koff(v16)
    B, H, Sq, Skv = x.shape
    if qtmem is None:
        qtmem = D == 256 and not v16
    nq = n_tiles_per_cta(D)
    rows_total = -(-Sq // (BM * nq)) * BM * nq
    pad = rows_total - Sq
    if pad:
        extra = np.repeat(x[:, :, -1:], pad, axis=2) if qtmem else np.zeros((B, H, pad, Skv))
        x = np.concatenate([x, extra], axis=2)
    nst_all = -(-Skv // BS)
    row = np.arange(rows_total)
    col = np.arange(Skv)
    vis = np.broadcast_to(col[None, :] < Skv, (rows_total, Skv)).copy()
    if causal:
        vis &= col[None, :] <= np.minimum(row, Skv - 1)[:, None]
    events, max_exp, steps = set(), -np.inf, 0
    for t0 in range(0, rows_total, BM):
        nst = min(nst_all, t0 // BS + 2) if causal else nst_all
        steps = max(steps, nst)
        xs = np.where(vis[None, None, t0:t0 + BM], x[:, :, t0:t0 + BM], -np.inf)  # [B,H,128,Skv]
        m_used = np.full((B, H, BM), -np.inf)
        for j in range(nst):
            s = xs[..., j * BS:(j + 1) * BS]
            mx = s.max(-1)
            if j == 0:
                m_used = mx
            else:
                grow = (mx - m_used) > tau                           # [B,H,128]
                need = grow.reshape(B, H, BM // WARP, WARP).any(-1)   # [B,H,4]
                for b, h, w in zip(*np.nonzero(need)):
                    events.add((int(b), int(h), int(t0 // WARP + w), j))
                need_rows = np.repeat(need, WARP, axis=-1)
                m_used = np.where(need_rows, np.maximum(m_used, mx), m_used)
            with np.errstate(invalid="ignore"):
                e = koff + s - m_used[..., None]
            fin = np.isfinite(e)
            if fin.any():
                max_exp = max(max_exp, float(e[fin].max()))
    return Replay(events=events, max_exp=max_exp, steps=steps)


def logsumexp_ref(x: np.ndarray, *, causal: bool) -> np.ndarray:
    """Natural-log sum-exp per row of the scores ``x`` (log2 units, sm_scale = ln 2), fp64 - what ``lse`` holds."""
    s = x * LN2
    if causal:
        Sq, Skv = x.shape[-2:]
        s = np.where(np.arange(Skv)[None, :] > np.arange(Sq)[:, None], -np.inf, s)
    m = s.max(-1, keepdims=True)
    return (m + np.log(np.exp(s - m).sum(-1, keepdims=True)))[..., 0]


def e4m3_lse_bound() -> float:
    """How far the single-e4m3 P mode's LSE may sit from the exact one: every p' it sums is rounded to e4m3, i.e.
    scaled by a factor in [1/(1 + 2^-4), 1 + 1/17], and the exponentials themselves carry up to ~2e-3."""
    return math.log1p(2.0**-4) + 2e-3


E4M3_P_HEADROOM = 2.0 ** (tau_koff(False)[0] + tau_koff(False)[1])  # 256 < 448


# ------------------------------------------------------------------------------------------------ the catalogue
def c4_tail(tau: float) -> Design:
    """For Skv = 75 600 (1 182 steps, the last one 16 keys): a staircase of six rescales over steps 1171-1176, then a
    jump in the 16-key last step."""
    d = tau + 0.25
    stairs = tuple((j * BS, (j - 1170) * d) for j in range(1171, 1177))
    return Design("c4_tail", sel_level=stairs + ((1181 * BS, 7 * d),))


@dataclass(frozen=True)
class Case:
    """One landscape run by tests/test_softmax_dynamics_gpu.py.  ``make(tau)`` builds the design for the TAU of the P
    mode (16-bit P: 8, e4m3 P: 4); ``expect`` lists the steps j >= 1 at which some warp must rescale."""
    name: str
    make: object
    D: int
    Sq: int
    Skv: int
    causal: bool
    expect: tuple


_EVERY = tuple(range(1, 16))
_EVEN = tuple(range(2, 16, 2))
CASES = [
    # both P-buffer / pv_done parities: j - 1 = 0, 1, 2
    Case("j1_above_d64", lambda t: jump(1, t + 0.25), 64, 1024, 1024, False, (1,)),
    Case("j2_above_d128_causal", lambda t: jump(2, t + 0.25), 128, 1000, 1000, True, (2,)),
    Case("j3_3tau_d256_causal", lambda t: jump(3, 3 * t), 256, 1024, 1024, True, (3,)),
    # headroom: a jump just under TAU takes no rescale and p' reaches 2^(KOFF + TAU - 1/8)
    Case("j1_below_d128", lambda t: jump(1, t - 0.25), 128, 1024, 1024, False, ()),
    Case("j5_below_d256_causal", lambda t: jump(5, t - 0.25), 256, 1000, 1000, True, ()),
    # past the K / V ring's first wrap (2 * STAGES steps), with a rescale that zeroes the past
    Case("j9_60_d64_causal", lambda t: jump(9, 60.0), 64, 1000, 1000, True, (9,)),
    Case("j9_60_d256", lambda t: jump(9, 60.0), 256, 1024, 1024, False, (9,)),
    # the last step, which is also the ragged 40-key tail step (masked tail instance of the step)
    Case("jlast_ragged_d256", lambda t: jump(15, t + 0.25), 256, 1000, 1000, False, (15,)),
    Case("jlast_ragged_d64", lambda t: jump(15, t + 0.25), 64, 1000, 1000, False, (15,)),
    Case("jlast_d128", lambda t: jump(15, t + 0.25), 128, 1024, 1024, False, (15,)),
    # one row per warp votes (lane 17); the other 31 rows take the rescale with alpha ~ 1
    Case("j14_lane17_d128", lambda t: jump(14, t + 0.25, "lane17"), 128, 1024, 1024, False, (14,)),
    Case("j2_lane17_d256_causal", lambda t: jump(2, 60.0, "lane17"), 256, 1024, 1024, True, (2,)),
    Case("j6_lane17_d64_causal", lambda t: jump(6, 3 * t, "lane17"), 64, 1000, 1000, True, (6,)),
    # the second query tile of a CTA alone; at causal step 11 its rows 704-767 rescale on the diagonal
    Case("j11_tile1_d128_causal", lambda t: jump(11, 3 * t, "tile1"), 128, 1000, 1000, True, (11,)),
    Case("j4_tile1_d64", lambda t: jump(4, t + 0.25, "tile1"), 64, 1024, 1024, False, (4,)),
    # a rescale at every step / at every other step
    Case("stairs_above_d64_causal", lambda t: staircase(t + 0.25, 0, 15), 64, 1024, 1024, True, _EVERY),
    Case("stairs_above_d128", lambda t: staircase(t + 0.25, 0, 15), 128, 1000, 1000, False, _EVERY),
    Case("stairs_above_d256_causal", lambda t: staircase(t + 0.25, 0, 15), 256, 1000, 1000, True, _EVERY),
    Case("stairs_below_d256", lambda t: staircase(t - 0.25, 0, 15), 256, 1000, 1000, False, _EVEN),
    Case("stairs_below_d128_causal", lambda t: staircase(t - 0.25, 0, 15), 128, 1024, 1024, True, _EVEN),
    Case("stairs_below_d64", lambda t: staircase(t - 0.25, 0, 15), 64, 1024, 1024, False, _EVEN),
    # p' of all but one key under the -125 clamp of the polynomial, MUFU's flush to zero and fp16's subnormals
    Case("descending_d64_causal", lambda t: descending(), 64, 1000, 1000, True, ()),
    Case("descending_d128", lambda t: descending(), 128, 1024, 1024, False, ()),
    Case("descending_d256", lambda t: descending(), 256, 1024, 1024, False, ()),
    # one key dominates its row at p' = 2^(KOFF + 3 + 5/64): the e4m3 rounding of p' moves the LSE by ~0.05
    Case("spike_d128", lambda t: spike(3, 3 + 5 / 64), 128, 1024, 1024, False, ()),
    Case("spike_d64_causal", lambda t: spike(1, 3 + 5 / 64), 64, 1000, 1000, True, ()),
]
LONG = Case("c4_tail", c4_tail, 128, 256, 75600, False, tuple(range(1171, 1177)) + (1181,))

# Causal problems with Sq != Skv (top-left mask: row i sees keys 0 .. min(i, Skv - 1)), run by
# tests/test_causal_rectangular_gpu.py.  RECT_WARPS: the 32-row warps that must rescale, where the design pins them.
RECT_CASES = [
    # level-60 keys from key 640 on, past every row's diagonal (rows < 512): no rescale, and a kernel that reads them
    # (a step too far, or a bottom-right mask) is off by orders of magnitude
    Case("rect_j10_60_512x2048_d128", lambda t: jump(10, 60.0), 128, 512, 2048, True, ()),
    # keys 256-319 (step 4) only reach rows >= 256: tiles 0 and 1 stop at 2 and 4 steps, warps 8-31 rescale
    Case("rect_j4_3tau_1024x320_d128", lambda t: jump(4, 3 * t), 128, 1024, 320, True, (4,)),
    Case("rect_j4_3tau_1024x320_d256", lambda t: jump(4, 3 * t), 256, 1024, 320, True, (4,)),
    # the ragged last step (keys 256-299 of 300): a spike that rows >= 261 see, and a jump that rows >= 256 see
    Case("rect_spike_ragged_1000x300_d64", lambda t: spike(4, 3 + 5 / 64), 64, 1000, 300, True, ()),
    Case("rect_jlast_ragged_1000x300_d256", lambda t: jump(4, t + 0.25), 256, 1000, 300, True, (4,)),
]
RECT_WARPS = {"rect_j4_3tau_1024x320_d128": range(8, 32), "rect_j4_3tau_1024x320_d256": range(8, 32),
              "rect_jlast_ragged_1000x300_d256": range(8, 32)}
