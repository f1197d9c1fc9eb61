"""Multi-GPU layouts of the FP8 attention path: one process per GPU, ``torch.distributed`` for the plumbing.

The reference is single-device (its launcher puts a DeviceGuard on q's device and launches on the current stream,
src/quantum_attn/tk/attention.py:417,465); callers such as ParaAttention shard the work around it.  Two layouts:

* **head sharding** - every (batch, head) is an independent problem (the kernel's grid y/z axes,
  src/quantum_attn/tk/attention.py:504; head-wise scales are per (b, h), src/quantum_attn/nn.py:411-412), so ranks
  take contiguous head ranges and there is NO collective: ``shard_heads`` / ``head_sharded_fp8_attention``.
* **sequence sharding** for shapes whose single (b, h) problems are too long for one GPU's share of the latency budget
  (BASELINE config 4, S = 75 600): each rank owns S/N tokens of Q, K and V.  Q and K (and V in the FP8 P modes) are
  quantised ONCE to e4m3 with head scales made global by a single ``all_reduce(MAX)`` (<= 12*B*H bytes) - so the bytes
  are the ones the unsharded call would produce, in EVERY P mode including the default "16bit" (e4m3 K and 16-bit V on
  the wire: the reference's numerics, inside the 2e-2 bound).  Strategy ``gather`` (default): the K / V blocks of
  all ranks are laid end to end PER HEAD in local memory, a few heads at a time, and each group of heads is attended
  in one launch over all keys as soon as its blocks are there - no partial results, no merge, no re-layout copy.  The
  blocks travel either by grouped NCCL all-gathers (``transport="nccl"``) or - ``transport="peer"`` - are PULLED from
  the other ranks' peer-mapped buffers by the copy engines (``qa_copy_2d``), which crosses NVSwitch without taking
  an SM from the attention kernel.  Strategy ``ring``: neighbour ``batch_isend_irecv`` while the fused kernel attends
  the block already here, partial results combined through their log-sum-exp by ``qa_merge_partials``.
  The gather strategy also serves GQA (only the Hkv heads of K / V travel) and causal attention over ZIG-ZAG shards:
  the sequence is cut into 2N chunks and rank r holds chunk r followed by chunk 2N-1-r (``zigzag_shard``), which gives
  every rank the same causal work.  K / V are gathered in global token order, and each head group is attended in two
  launches - one per local chunk - whose causal diagonal sits at the END of the keys that chunk sees (the
  bottom-right alignment of the C ABI, QA_CAUSAL_BOTTOM_RIGHT).  The ring strategy is non-causal and MHA only.

The kernels are reached through a small backend object so that the host logic (ring order, buffer rotation, scale
exchange, merge order) can be exercised on CPU with the ``gloo`` backend in tests; the default backend is the
sm_100a library and has no fallback.
"""
from __future__ import annotations

import math
import os
from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import _native, ops


# ------------------------------------------------------------------------------------------------ head sharding
def shard_heads(n_heads: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous head range [start, stop) of ``rank``; the first ``n_heads % world_size`` ranks take one extra."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError(f"bad rank {rank} for world size {world_size}")
    base, extra = divmod(n_heads, world_size)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def head_sharded_fp8_attention(q, k, v, *, is_causal=False, scale=None, scaling_method="head-wise", group=None,
                               gather: bool = False, _attn=None):
    """Run this rank's head range of a replicated [B,H,S,D] problem; no collective unless ``gather`` asks for the
    full output back (one all_gather of the outputs; head counts must then divide evenly)."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    Hq, Hkv = q.shape[1], k.shape[1]
    if Hq % Hkv:
        raise ValueError(f"Expect Hq to be a multiple of Hkv but got Hq={Hq} and Hkv={Hkv}.")
    lo, hi = shard_heads(Hkv, world, rank)  # shard KV heads so that GQA groups stay together
    g = Hq // Hkv
    if _attn is None:
        from . import nn as _nn

        def _attn(q_, k_, v_):
            return _nn.fp8_attention(q_, k_, v_, is_causal=is_causal, scale=scale, scaling_method=scaling_method)
    if hi > lo:
        out = _attn(q[:, lo * g:hi * g], k[:, lo:hi], v[:, lo:hi])
    else:
        out = q.new_empty((q.shape[0], 0, q.shape[2], q.shape[3]))
    if not gather:
        return out
    if Hkv % world:
        raise ValueError("gather=True needs the head count to divide evenly over the ranks")
    parts = [torch.empty_like(out) for _ in range(world)]
    dist.all_gather(parts, out.contiguous(), group=group)
    return torch.cat(parts, dim=1)


# ------------------------------------------------------------------------------------------------ sequence sharding
class NativeBackend:
    """The sm_100a kernels (include/qattn.h).  Raises if the library or the device is missing."""

    def local_scales(self, tensors: Sequence[torch.Tensor]) -> List[torch.Tensor]:
        _, scales = _native.quantize_fp8(list(tensors), _native.QA_SCALE_HEAD_AMAX_ONLY)
        return scales

    def quantize(self, tensors: Sequence[torch.Tensor], scales: Sequence[torch.Tensor], outs=None) -> List[torch.Tensor]:
        outs, _ = _native.quantize_fp8(list(tensors), _native.QA_SCALE_HEAD_GIVEN, scales=list(scales), outs=outs)
        return outs

    def attend(self, q8, k8, v, sq, sk, sv, sm_scale, p_mode, out_dtype, out=None, return_lse=True, gate=None, causal=0):
        """``causal``: 0, QA_CAUSAL_TOP_LEFT or QA_CAUSAL_BOTTOM_RIGHT (include/qattn.h)."""
        return _native.fp8_attn_fwd(q8, k8, v, sq, sk, sv, scale_mode=_native.QA_SCALE_HEAD, is_causal=causal,
                                    sm_scale=sm_scale, p_mode=p_mode, out_dtype=out_dtype, return_lse=return_lse, out=out,
                                    gate=gate)

    def merge(self, o_acc, lse_acc, o_new, lse_new, first, out=None):
        _native.merge_partials(o_acc, lse_acc, o_new, lse_new, first=first, out=out)


def _ring_exchange(send_buf: torch.Tensor, recv_buf: torch.Tensor, group) -> list:
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    nxt = dist.get_global_rank(group, (rank + 1) % world) if group is not None else (rank + 1) % world
    prv = dist.get_global_rank(group, (rank - 1) % world) if group is not None else (rank - 1) % world
    ops_ = [dist.P2POp(dist.isend, send_buf, nxt, group), dist.P2POp(dist.irecv, recv_buf, prv, group)]
    return dist.batch_isend_irecv(ops_)


# bench.py's time split: set to a list to collect (label, CUDA event) marks on the calling stream at the phase
# boundaries of ring_fp8_attention (gather strategy); None (default) records nothing
trace_marks = None


def _mark(label: str, device) -> None:
    if trace_marks is not None:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(device))
        trace_marks.append((label, ev))


SEQ_STRATEGIES = ("gather", "ring")
SEQ_TRANSPORTS = ("auto", "nccl", "peer")


def zigzag_shard(x: torch.Tensor, world: int, rank: int) -> torch.Tensor:
    """Rank ``rank``'s shard of a global [B, H, S, D] sequence for causal sequence sharding: dim 2 cut into 2 * world
    chunks of c = S / (2 * world) tokens, rank r holding chunk r followed by chunk 2 * world - 1 - r ([B, H, 2c, D]).
    Row i of a causal problem attends i + 1 keys, so chunk j costs ~ (j + 1/2) c^2 and every rank's pair of chunks
    costs the same 2 * world * c^2."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"bad rank {rank} for world size {world}")
    S = x.shape[2]
    if S % (2 * world):
        raise ValueError(f"zigzag_shard: the sequence length {S} must be a multiple of 2 * world = {2 * world}")
    c = S // (2 * world)
    return torch.cat([x[:, :, rank * c:(rank + 1) * c], x[:, :, (2 * world - 1 - rank) * c:(2 * world - rank) * c]], 2)


def zigzag_unshard(shards: Sequence[torch.Tensor]) -> torch.Tensor:
    """Inverse of ``zigzag_shard``: the [B, H, 2c, D] shards of ranks 0 .. N-1 -> the global [B, H, 2Nc, D] sequence."""
    world = len(shards)
    c = shards[0].shape[2] // 2
    chunks = [None] * (2 * world)
    for r, t in enumerate(shards):
        if t.shape[2] != 2 * c:
            raise ValueError("zigzag_unshard: every shard must have the same even length")
        chunks[r], chunks[2 * world - 1 - r] = t[:, :, :c], t[:, :, c:]
    return torch.cat(chunks, 2)


def seq_pv_mode() -> str:
    """P mode of the sequence-sharded path when the caller names none: the configured one - by default "16bit", the
    reference's numerics (e4m3 K and 16-bit V travel), which meets the 2e-2 max-abs bound like the one-GPU call."""
    from . import config

    return config.attention.pv_mode


def default_seq_strategy() -> str:
    """``QA_SEQ_STRATEGY`` (gather | ring), else the measured choice (DESIGN.md section 7)."""
    s = os.environ.get("QA_SEQ_STRATEGY", "gather")
    if s not in SEQ_STRATEGIES:
        raise ValueError(f"QA_SEQ_STRATEGY must be one of {SEQ_STRATEGIES} but got {s!r}")
    return s


def default_seq_transport() -> str:
    """``QA_SEQ_TRANSPORT`` (auto | nccl | peer), else "auto": copy-engine pulls from peer-mapped symmetric memory
    where the ranks can map each other's buffers (measured on two B200s, C4: 24.1 ms against 24.7 ms with NCCL
    all-gathers, whose kernels take SMs from the attention kernel), NCCL otherwise."""
    s = os.environ.get("QA_SEQ_TRANSPORT", "auto")
    if s not in SEQ_TRANSPORTS:
        raise ValueError(f"QA_SEQ_TRANSPORT must be one of {SEQ_TRANSPORTS} but got {s!r}")
    return s


def seq_gated_launch(B: int = 1, H: int = 1 << 20, S_local: int = 1 << 20, n_sms: int = 148) -> bool:
    """Should the gather strategy (peer transport) attend ALL heads in ONE gated launch (``qa_fp8_attn_fwd_gated``: the
    CTAs of a head group poll a flag its copies set) instead of one launch per head group?  Per-group launches run in
    lock-step - each waits for the slowest CTA of the one before - while one launch lets fast SMs take more CTAs; that
    only pays when an SM gets enough CTAs per call to balance with.  Measured on C4 (strong-scaling efficiency, gated
    against per-group): N = 4 (12 CTAs per SM) 0.974 / 0.950; N = 8 (6 per SM) 0.923 / 0.954.  ``QA_SEQ_GATED`` = 1 / 0
    forces it on / off; default: on from 8 CTAs per SM."""
    env = os.environ.get("QA_SEQ_GATED", "auto")
    if env in ("0", "1"):
        return env == "1"
    return B * H * ((S_local + 255) // 256) >= 8 * n_sms


_peer_unavailable = {}  # id(group) -> reason the peer transport could not be set up (then "auto" means NCCL)


def resolve_transport(transport: str, group, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, v_itemsize: int):
    """-> ("peer", PeerGather) or ("nccl", None).  "auto" tries the peer transport once per group; setting it up is a
    collective (a symmetric-memory rendezvous), so every rank takes the same branch."""
    if transport == "nccl" or not q.is_cuda:
        return "nccl", None
    key = id(group) if group is not None else 0
    if transport == "auto" and key in _peer_unavailable:
        return "nccl", None
    try:
        return "peer", PeerGather.get(group, q.device, k.shape, v.shape, v_itemsize)
    except Exception as e:
        if transport == "peer":
            raise
        _peer_unavailable[key] = repr(e)[:200]
        return "nccl", None


def last_transport_error(group=None):
    return _peer_unavailable.get(id(group) if group is not None else 0)


def head_chunks(B: int, H: int, S_local: int, n_sms: int = 148, max_chunks: int = 12) -> List[Tuple[int, int]]:
    """Head ranges [lo, hi) the gather strategy moves and attends one after the other.  A launch over ``hc`` heads has
    B * hc * ceil(S_local / 256) CTAs (two 128-row query tiles per CTA, one CTA per SM).  ``hc`` is the SMALLEST head
    count (most groups, so the transfer of group i + 1 hides under the attention of group i and the exposed first
    transfer is short) among those whose launch wastes the least of its last wave - no launch then pays more wave
    quantisation than a single launch over all heads would.  At most ``max_chunks`` groups.

    ``ring_fp8_attention`` passes the kv heads as ``H`` and B * (Hq / Hkv) as ``B`` (a group of kv heads attends all
    their query heads in one launch).  Causal calls pass S_local / 2: a group is attended in two launches of one zig-zag
    chunk each, which have the same CTA count; their CTAs do different work (rank r's first chunk sees (r + 1) chunks of
    keys, its second 2N - r), so the sizing fills the waves by CTA count only, as it does for the causal diagonal
    inside any one launch."""
    ctas_per_head = max(1, B * ((S_local + 255) // 256))
    best = None
    for hc in range(1, H + 1):
        if -(-H // hc) > max_chunks:
            continue
        n = hc * ctas_per_head
        waste = round((-(-n // n_sms) * n_sms) / n, 2)  # SM-slots paid per SM-slot used (1.0 = whole waves)
        if best is None or waste < best[0]:
            best = (waste, hc)
    hc = best[1] if best else H
    return [(lo, min(H, lo + hc)) for lo in range(0, H, hc)]


class _Works:
    """wait() on a set of async collectives (one coalesced work, or several plain ones)."""

    def __init__(self, works):
        self.works = [w for w in works if w is not None]

    def wait(self):
        for w in self.works:
            w.wait()


def _nccl_gather_heads(srcs: Sequence[torch.Tensor], dsts: Sequence[torch.Tensor], lo: int, hi: int, group) -> _Works:
    """All-gather heads [lo, hi) of every ``src`` [B,H,S,*] into ``dst`` [B,H,world*S,*]: per (b, h) the blocks of all
    ranks end to end in rank order.  One all-gather per (tensor, b, h) - each a contiguous S x row chunk on both
    sides - issued as ONE grouped NCCL call where the backend can coalesce them."""
    pairs = []
    for src, dst in zip(srcs, dsts):
        for b in range(src.shape[0]):
            for h in range(lo, hi):
                pairs.append((dst[b, h].view(torch.uint8), src[b, h].view(torch.uint8)))
    if srcs[0].is_cuda:
        with dist._coalescing_manager(group=group, async_ops=True) as cm:
            for o, i in pairs:
                dist.all_gather_into_tensor(o, i, group=group)
        return _Works([cm])
    # (gloo, CPU tests: no coalesced all-gather; same data movement, one collective each)
    return _Works([dist.all_gather_into_tensor(o, i, group=group, async_op=True) for o, i in pairs])


class PeerGather:
    """Copy-engine gather over NVSwitch peer memory.  Every rank keeps its outgoing K / V blocks in a symmetric-memory
    buffer (mapped into every peer's address space through CUDA IPC by ``torch.distributed._symmetric_memory``); after
    a device-side barrier each rank PULLS the other ranks' blocks into its own per-head layout with strided copies on
    a side stream (``qa_copy_2d``: cudaMemcpy2DAsync from the peer pointer).  No kernel is launched for the transfer.
    Two send slots alternate so that one barrier per call suffices: a peer still reading slot p of call i has finished
    before it reaches the barrier of call i + 1, and slot p is next written in call i + 2."""

    _cache = {}

    @classmethod
    def get(cls, group, device, k_shape, v_shape, v_itemsize):
        key = (id(group) if group is not None else 0, device.index, tuple(k_shape), tuple(v_shape), v_itemsize)
        obj = cls._cache.get(key)
        if obj is None:
            obj = cls._cache[key] = cls(group, device, k_shape, v_shape, v_itemsize)
        return obj

    def __init__(self, group, device, k_shape, v_shape, v_itemsize):
        import torch.distributed._symmetric_memory as symm_mem

        pg = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(pg), dist.get_rank(pg)
        self.device = device
        self.nk = int(torch.Size(k_shape).numel())
        self.nv = int(torch.Size(v_shape).numel()) * v_itemsize
        self.slot = (self.nk + self.nv + 255) // 256 * 256
        try:
            symm_mem.enable_symm_mem_for_group(pg.group_name)
        except Exception:
            pass
        self.buf = symm_mem.empty(2 * self.slot, dtype=torch.uint8, device=device)
        self.hdl = symm_mem.rendezvous(self.buf, pg)
        self.peers = [self.hdl.get_buffer(r, (2 * self.slot,), torch.uint8, 0) for r in range(self.world)]
        self.peer_ptrs = [t.data_ptr() for t in self.peers]
        self.streams = [torch.cuda.Stream(device=device) for _ in range(int(os.environ.get("QA_PEER_STREAMS", "2")))]
        self.batches = {}
        self.cur = 0
        self.phase = 0
        B, H, S, D = k_shape
        # gated launch: one word per (head group, copy stream), set behind the group's copies on that stream
        self.flags = torch.zeros((64 * len(self.streams),), dtype=torch.int32, device=device)
        self.k_all = torch.empty((B, H, self.world * S, D), dtype=torch.uint8, device=device)
        self.v_all = torch.empty((B, H, self.world * S, D * v_itemsize), dtype=torch.uint8, device=device)

    def send_views(self, k_shape, v_shape, v_itemsize):
        """This call's slot of the local symmetric buffer as (k8 bytes [B,H,S,D], v bytes [B,H,S,D*itemsize])."""
        base = self.phase * self.slot
        kb = self.buf[base:base + self.nk].view(k_shape)
        vb = self.buf[base + self.nk:base + self.nk + self.nv].view(tuple(v_shape[:-1]) + (v_shape[-1] * v_itemsize,))
        return kb, vb

    def start(self) -> None:
        """Device-side barrier (every rank's blocks of this call are in its slot); the copy streams wait for it."""
        main = torch.cuda.current_stream(self.device)
        self.hdl.barrier(channel=self.phase)
        ready = torch.cuda.Event()
        ready.record(main)
        for st in self.streams:
            st.wait_event(ready)
        self.cur, self.phase = self.phase, self.phase ^ 1

    def pull_group(self, lo: int, hi: int, gate_index: Optional[int] = None, zigzag: bool = False) -> List[torch.cuda.Event]:
        """Start the pulls of heads [lo, hi) from every rank (own block: a local copy); returns the events to wait for -
        or, with ``gate_index``, sets the group's words of ``self.flags`` behind the copies instead (gated launch).
        The copies are dealt round-robin to a few streams so that transfers from different peers overlap; the argument
        arrays of a (slot, head range) are marshalled once and re-issued with one call of the C ABI - the host cost of
        issuing the copies is what the first head group's transfer hides behind, so it has to be small.
        ``zigzag``: the blocks are zig-zag shards (``zigzag_shard``), and their two halves go to their places in global
        token order - two copy rows per rank-block."""
        key = (self.cur, lo, hi, gate_index is not None, zigzag)
        batch = self.batches.get(key)
        if batch is None:
            B, H, S_all, D = self.k_all.shape
            S = S_all // self.world
            Dv = self.v_all.shape[-1]
            base = self.cur * self.slot
            k_dst, v_dst = self.k_all.data_ptr(), self.v_all.data_ptr()
            raws = [st.cuda_stream for st in self.streams]
            copies, n = [], 0
            # (gated launch: the own block is NOT pulled here - a device-local 2-D copy is a kernel, and no kernel can run
            # while the polling attention launch holds every SM; fill_own() puts it in place before the launch.  Copies
            # from PEER memory run on the copy engines: scripts/gate_probe.py)
            for i in range(1 if gate_index is not None else 0, self.world):
                r = (self.rank + i) % self.world  # own block first, then the peers - every rank in another order
                src = self.peer_ptrs[r] + base
                # (first row of the block, first row in the per-head layout, rows): the whole block at r * S, or its
                # zig-zag halves at chunks r and 2N - 1 - r
                c = S // 2
                segs = [(0, r * c, c), (c, (2 * self.world - 1 - r) * c, c)] if zigzag else [(0, r * S, S)]
                for s0, d0, rows in segs:
                    for b in range(B):
                        # rows = heads of the group; a row is this rank-block of one head: rows x D bytes of K, x Dv of V
                        copies.append((k_dst + ((b * H + lo) * S_all + d0) * D, S_all * D,
                                       src + ((b * H + lo) * S + s0) * D, S * D, rows * D, hi - lo, raws[n % len(raws)]))
                        copies.append((v_dst + ((b * H + lo) * S_all + d0) * Dv, S_all * Dv,
                                       src + self.nk + ((b * H + lo) * S + s0) * Dv, S * Dv, rows * Dv, hi - lo,
                                       raws[(n + 1) % len(raws)]))
                        n += 2
            batch = self.batches[key] = _native.CopyBatch(copies)
        batch.issue()
        if gate_index is not None:
            for i, st in enumerate(self.streams):
                _native.set_flag(self.flags, gate_index * len(self.streams) + i, st.cuda_stream)
            return []
        evs = []
        for st in self.streams:
            ev = torch.cuda.Event()
            ev.record(st)
            evs.append(ev)
        return evs

    def fill_own(self, kb: torch.Tensor, vb: torch.Tensor) -> None:
        """This rank's own blocks (all heads) into their place in the per-head layout, on the calling stream."""
        B, H, S_all, D = self.k_all.shape
        S, Dv = S_all // self.world, self.v_all.shape[-1]
        raw = torch.cuda.current_stream(self.device).cuda_stream
        # one strided copy per tensor: row (b, h) = this rank's S x D bytes, S_all x D apart in the per-head layout
        _native.copy_2d(self.k_all.data_ptr() + self.rank * S * D, S_all * D, kb.data_ptr(), S * D, S * D, B * H, raw)
        _native.copy_2d(self.v_all.data_ptr() + self.rank * S * Dv, S_all * Dv, vb.data_ptr(), S * Dv, S * Dv, B * H, raw)

    def pull(self, chunks: Sequence[Tuple[int, int]]) -> List[List[torch.cuda.Event]]:
        """start() + every head group at once (bench.py's transfer-alone probe)."""
        self.start()
        return [self.pull_group(lo, hi) for lo, hi in chunks]


def ring_fp8_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, is_causal: bool = False,
                       scale: Optional[float] = None, pv_mode: Optional[str] = None, group=None, backend=None,
                       strategy: Optional[str] = None, transport: Optional[str] = None,
                       head_groups: Optional[int] = None) -> torch.Tensor:
    """FP8 attention over a sequence sharded across the ranks of ``group``.

    q, k, v: this rank's [B, Hq, S_local, D] / [B, Hkv, S_local, D] 16-bit slices (equal S_local on every rank;
    Hq = Hkv with the ring strategy, a multiple of it with the gather strategy); returns the [B, Hq, S_local, D] output
    rows of the local queries against the keys/values of ALL ranks.  Non-causal: the slices are contiguous shards of
    the sequence (rank r holds tokens [r * S_local, (r + 1) * S_local)).  ``is_causal``: the slices are ZIG-ZAG shards
    (``zigzag_shard``; S_local even), each local query attends the keys up to its own global position (top-left
    causal attention over the whole sequence), and the output rows come back in the same zig-zag order
    (``zigzag_unshard`` reassembles the sequence).  With world size 1 this is exactly ``fp8_attn_func(q, k, v,
    is_causal=is_causal)`` in the chosen P mode (the configured one when none is given; every mode is supported: in
    "16bit" the value blocks travel in 16 bits).

    ``strategy`` "gather" (default): per group of heads, all ranks' K / V blocks are laid end to end in local memory
    and attended in ONE launch over all keys - no partial results; group i + 1 travels while group i is attended.
    ``transport`` chooses how they travel: "nccl" (grouped all-gathers) or "peer" (copy-engine pulls from peer-mapped
    symmetric memory; no SM is spent on communication).  ``head_groups`` overrides the number of head groups
    (default: ``head_chunks``).  ``strategy`` "ring": world - 1 neighbour exchanges, one launch and one (O, LSE) merge
    per block.  Same quantised bytes every way.

    Causal calls (gather strategy only): K / V are laid out in global token order, and each head group is attended in
    two launches, one per local chunk, against the keys up to that chunk's end - (r + 1) c and (2N - r) c keys for
    chunk size c = S_local / 2 - with the causal diagonal aligned to the last key (QA_CAUSAL_BOTTOM_RIGHT).  They use
    per-group launches synchronised by events, never the gated launch.
    """
    be = backend if backend is not None else NativeBackend()
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    strategy = default_seq_strategy() if strategy is None else strategy
    if strategy not in SEQ_STRATEGIES:
        raise ValueError(f"strategy must be one of {SEQ_STRATEGIES} but got {strategy!r}")
    if strategy == "ring":
        if q.dim() != 4 or k.shape != v.shape or q.shape[:2] != k.shape[:2] or q.shape[3] != k.shape[3]:
            raise ValueError("ring_fp8_attention: q, k, v must be [B,H,S_local,D] with equal B, H, D (no GQA)")
        if is_causal:
            raise ValueError("ring_fp8_attention: the ring strategy is non-causal only; use strategy='gather'")
    elif (q.dim() != 4 or k.dim() != 4 or k.shape != v.shape or q.shape[0] != k.shape[0] or q.shape[2:] != k.shape[2:]
          or q.shape[1] % k.shape[1]):
        raise ValueError("ring_fp8_attention: q, k, v must be [B,Hq,S_local,D], [B,Hkv,S_local,D] with Hq a multiple "
                         "of Hkv")
    if is_causal and world > 1 and q.shape[2] % 2:
        raise ValueError(f"ring_fp8_attention: a causal zig-zag shard holds two equal chunks, so S_local must be even "
                         f"(got {q.shape[2]})")
    if pv_mode is None:
        pv_mode = seq_pv_mode()
    p_mode = ops.pv_mode_code(pv_mode)
    v16 = p_mode == _native.QA_P_16BIT
    transport = default_seq_transport() if transport is None else transport
    if transport not in SEQ_TRANSPORTS:
        raise ValueError(f"transport must be one of {SEQ_TRANSPORTS} but got {transport!r}")
    B, Hq, S, D = q.shape
    H = k.shape[1]  # kv heads: what travels, and what head groups are made of
    g = Hq // H     # query heads per kv head (GQA): group [lo, hi) attends query heads [lo * g, hi * g)
    sm_scale = (1.0 / math.sqrt(D)) if scale is None else float(scale)

    # 1. head scales of the WHOLE sequence: local scales, one MAX all-reduce (scale is monotone in amax) over the
    #    [B,Hq] and [B,Hkv] scales laid end to end
    if q.is_cuda:
        _mark("start", q.device)
    kv_in = [k] if v16 else [k, v]
    local = be.local_scales([q] + kv_in) if g == 1 else be.local_scales([q]) + be.local_scales(kv_in)
    scales = torch.cat([t.reshape(-1) for t in local])  # fp32 [B*Hq + (1 or 2) * B*Hkv]
    if q.is_cuda:
        _mark("amax", q.device)
    if world > 1:
        dist.all_reduce(scales, op=dist.ReduceOp.MAX, group=group)
    n_sq, n_sk = B * Hq, B * H
    sq, sk = scales[:n_sq].view(B, Hq), scales[n_sq:n_sq + n_sk].view(B, H)
    sv = None if v16 else scales[n_sq + n_sk:].view(B, H)
    out = torch.empty_like(q)
    if q.is_cuda:
        _mark("scales", q.device)
    causal_kw = {"causal": _native.QA_CAUSAL_TOP_LEFT} if is_causal else {}

    if world == 1:
        if g == 1:
            q8, k8 = be.quantize([q, k], [sq, sk])
        else:
            (q8,), (k8,) = be.quantize([q], [sq]), be.quantize([k], [sk])
        v_in = v if v16 else be.quantize([v], [sv])[0]
        be.attend(q8, k8, v_in, sq, sk, sv, sm_scale, p_mode, q.dtype, out=out, return_lse=False, **causal_kw)
        return out

    if strategy == "gather":
        # 2. K / V first - they travel - then Q while the first blocks are on the wire
        c = S // 2 if is_causal else S  # query rows per launch
        if head_groups is None:
            chunks = head_chunks(B * g, H, c)
        else:  # caller's choice (tests; tuning)
            hc = -(-H // max(1, min(H, int(head_groups))))
            chunks = [(lo, min(H, lo + hc)) for lo in range(0, H, hc)]
        f8 = torch.float8_e4m3fn
        transport, comm = resolve_transport(transport, group, q, k, v, v.element_size() if v16 else 1)
        main = torch.cuda.current_stream(q.device) if q.is_cuda else None
        if transport == "peer":
            kb, vb = comm.send_views(k.shape, v.shape, v.element_size() if v16 else 1)
            if v16:
                be.quantize([k], [sk], outs=[kb])
                vb.view(v.dtype).copy_(v)
            else:
                be.quantize([k, v], [sk, sv], outs=[kb, vb])
            # (causal: per-group launches - the two chunks of a group need launches of their own)
            gated = not is_causal and seq_gated_launch(B * g, H, S) and len(chunks) <= 64
            if gated:
                comm.flags.zero_()  # (on the calling stream, ahead of the event the copy streams wait for)
            comm.start()
            k_all = comm.k_all.view(f8)
            v_all = comm.v_all.view(v.dtype if v16 else f8)
            if gated:
                # ONE launch over all heads; the copies of head group g set the group's flags behind them and the CTAs of
                # its heads wait for those.  The first group's copies go out before Q is quantised, the launch follows,
                # and the host issues the later groups' copies while the kernel already runs.
                hc = chunks[0][1] - chunks[0][0]
                comm.pull_group(*chunks[0], gate_index=0)
                comm.fill_own(kb, vb)  # (kernels on this stream, under the first group's transfer)
                _mark("quant_kv", q.device)
                (q8,) = be.quantize([q], [sq])
                _mark("quant_q", q.device)
                dst = out if out.is_contiguous() else None
                o = be.attend(q8, k_all, v_all, sq, sk, None if v16 else sv, sm_scale, p_mode, q.dtype, out=dst,
                              return_lse=False, gate=(comm.flags, hc, len(comm.streams)))
                for i in range(1, len(chunks)):
                    comm.pull_group(*chunks[i], gate_index=i)
                if dst is None:
                    out.copy_(o)
                _mark("attend", q.device)
                return out
            fetch = lambda lo, hi: comm.pull_group(lo, hi, zigzag=is_causal)

            def wait(evs):
                for ev in evs:
                    main.wait_event(ev)
        else:
            if v16:
                (k8,) = be.quantize([k], [sk])
                v_send = v.contiguous()
            else:
                k8, v_send = be.quantize([k, v], [sk, sv])
            k_all = torch.empty((B, H, world * S, D), dtype=f8, device=q.device)
            v_all = torch.empty((B, H, world * S, D), dtype=v_send.dtype, device=q.device)
            if not is_causal:
                fetch = lambda lo, hi: _nccl_gather_heads([k8, v_send], [k_all, v_all], lo, hi, group)
                wait = lambda w: w.wait()
            else:
                # zig-zag halves: the first halves (chunks 0 .. N-1) land in rank order straight in place; the second
                # halves (chunk 2N-1-r of rank r) arrive in rank order, i.e. reversed, in a side buffer and are put in
                # place by one strided copy per tensor (index_copy_ with the reversed rank order) once they are there
                tails = [torch.empty((B, H, world * c, D), dtype=t.dtype, device=q.device) for t in (k8, v_send)]
                rev = torch.arange(world - 1, -1, -1, device=q.device)

                def fetch(lo, hi):
                    return lo, hi, _nccl_gather_heads(
                        [k8[:, :, :c], v_send[:, :, :c], k8[:, :, c:], v_send[:, :, c:]],
                        [k_all[:, :, :world * c], v_all[:, :, :world * c]] + tails, lo, hi, group)

                def wait(pending):
                    lo, hi, w = pending
                    w.wait()
                    for dst, tail in zip((k_all, v_all), tails):  # (as bytes: index_copy_ has no float8 kernels)
                        dst[:, lo:hi, world * c:].view(torch.uint8).view(B, hi - lo, world, c, -1).index_copy_(
                            2, rev, tail[:, lo:hi].view(torch.uint8).view(B, hi - lo, world, c, -1))
        # the first group's transfer is started at once; every later one right before the attention of the group in
        # front of it is launched, so the host never spends more than one group's worth of issue time ahead of a launch
        pending = fetch(*chunks[0])
        if q.is_cuda:
            _mark("quant_kv", q.device)
        (q8,) = be.quantize([q], [sq])
        if q.is_cuda:
            _mark("quant_q", q.device)
        # 3. one launch per head group over ALL keys (causal: two, one per zig-zag chunk), as its blocks land
        for i, (lo, hi) in enumerate(chunks):
            nxt = fetch(*chunks[i + 1]) if i + 1 < len(chunks) else None
            wait(pending)
            pending = nxt
            if q.is_cuda:
                _mark("wait", q.device)
            qh = slice(lo * g, hi * g)
            sv_g = None if v16 else sv[:, lo:hi]
            if not is_causal:
                dst = out[:, qh] if B == 1 else None  # (a head range of a [1,H,S,D] tensor is dense)
                o = be.attend(q8[:, qh], k_all[:, lo:hi], v_all[:, lo:hi], sq[:, qh], sk[:, lo:hi], sv_g, sm_scale,
                              p_mode, q.dtype, out=dst, return_lse=False)
                if dst is None:
                    out[:, qh].copy_(o)
            else:
                # chunk r sees the keys of chunks 0 .. r, chunk 2N-1-r those of chunks 0 .. 2N-1-r: each the keys up to
                # its own end, diagonal at the last key.  The kernel writes dense rows; a chunk of a head is not, so
                # its c x D output is copied into place.
                for rows, n_keys in ((slice(0, c), (rank + 1) * c), (slice(c, S), (2 * world - rank) * c)):
                    o = be.attend(q8[:, qh, rows], k_all[:, lo:hi, :n_keys], v_all[:, lo:hi, :n_keys], sq[:, qh],
                                  sk[:, lo:hi], sv_g, sm_scale, p_mode, q.dtype, return_lse=False,
                                  causal=_native.QA_CAUSAL_BOTTOM_RIGHT)
                    out[:, qh, rows].copy_(o)
            if q.is_cuda:
                _mark("attend", q.device)
        return out

    # strategy "ring": K and V share one byte buffer so a ring step is one send and one receive
    q8, k8 = be.quantize([q, k], [sq, sk])
    v_send = v.contiguous() if v16 else be.quantize([v], [sv])[0]
    nk, nv = k8.numel(), v_send.numel() * v_send.element_size()
    kv = [torch.empty((nk + nv,), dtype=torch.uint8, device=q.device) for _ in range(2)]
    kv[0][:nk].copy_(k8.view(torch.uint8).reshape(-1))
    kv[0][nk:].copy_(v_send.view(torch.uint8).reshape(-1))
    o_acc = torch.empty((B, H, S, D), dtype=torch.float32, device=q.device)
    lse_acc = torch.empty((B, H, S), dtype=torch.float32, device=q.device)
    cur = 0
    for step in range(world):
        last = step == world - 1
        # 3. start moving the block we hold to the next rank, then compute on it (the transfer only reads it)
        reqs = _ring_exchange(kv[cur], kv[cur ^ 1], group) if not last else []
        k_blk = kv[cur][:nk].view(torch.float8_e4m3fn).view(k8.shape)
        v_blk = kv[cur][nk:].view(v_send.dtype).view(v_send.shape)
        o_new, lse_new = be.attend(q8, k_blk, v_blk, sq, sk, sv, sm_scale, p_mode, q.dtype)
        # 4. fold the partial result in; the last step writes the 16-bit output directly
        be.merge(o_acc, lse_acc, o_new, lse_new, step == 0, out if last else None)
        for r in reqs:
            r.wait()
        cur ^= 1
    return out


# the function predates the gather strategy; this is the name that says what it does
sequence_sharded_fp8_attention = ring_fp8_attention


def ring_block_owner(rank: int, step: int, world: int) -> int:
    """Rank whose K/V block ``rank`` holds at ring step ``step`` (blocks travel to rank + 1 each step)."""
    return (rank - step) % world
