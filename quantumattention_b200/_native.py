"""ctypes binding of the C ABI in include/qattn.h.  PyTorch only supplies device memory and the current stream.

There is NO fallback: if the shared library is missing or the device is not sm_100 the calls raise.
"""
from __future__ import annotations

import contextlib
import ctypes
import os
import threading
from typing import Optional, Sequence, Tuple

import torch

from . import build as _build

QA_DT_BF16, QA_DT_FP16, QA_DT_E4M3 = 0, 1, 2
QA_SCALE_HEAD, QA_SCALE_TOKEN, QA_SCALE_HEAD_TWO_PASS, QA_SCALE_HEAD_AMAX_ONLY, QA_SCALE_HEAD_GIVEN = 0, 1, 2, 3, 4
QA_SCALE_HEAD_RELOAD = 5
QA_WS_PERSISTENT = 0x100  # qa_quantize_fp8: the workspace was zeroed once and is reused (include/qattn.h)
QA_P_E4M3, QA_P_E4M3_HILO, QA_P_16BIT = 0, 1, 2
QA_CAUSAL_TOP_LEFT, QA_CAUSAL_BOTTOM_RIGHT = 1, 2  # the `causal` argument of the attention entries (0: no mask)
ABI_VERSION = 7

EXPORTED_SYMBOLS = (
    "qa_abi_version",
    "qa_last_error",
    "qa_device_supported",
    "qa_quantize_workspace_floats",
    "qa_quantize_fp8",
    "qa_fp8_attn_fwd",
    "qa_fp8_attn_fwd_gated",
    "qa_set_flag",
    "qa_fp8_attn_func",
    "qa_attn_fwd",
    "qa_merge_partials",
    "qa_copy_2d",
    "qa_copy_2d_batch",
    "qa_last_launch_count",
)

_lib = None
_lock = threading.Lock()

# bookkeeping for bench.py: kernels launched through this binding, and an optional CUDA-event timer around the
# attention kernel (events are recorded on the launching stream; a few hundred ns each)
launch_total = 0
attn_events = None  # set to a list to collect (start_event, stop_event) pairs
quant_events = None  # the same for the quantiser launches


class NativeError(RuntimeError):
    pass


def lib_path() -> str:
    # QA_NATIVE_LIB: developer override to A/B kernel variants built by scripts/build_variant.sh
    return os.environ.get("QA_NATIVE_LIB") or _build.LIB_PATH


def load(build_if_missing: bool = True):
    """Load (building first if the .so is absent and nvcc is available).  Raises if it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = lib_path()
        if not os.path.exists(path):
            if not build_if_missing:
                raise NativeError(f"{path} is missing; run `python -m quantumattention_b200.build`")
            _build.build_library()  # (takes an inter-process lock: one rank builds, the others wait and re-check)
        lib = ctypes.CDLL(path)
        lib.qa_abi_version.restype = ctypes.c_int
        lib.qa_last_error.restype = ctypes.c_char_p
        lib.qa_last_launch_count.restype = ctypes.c_int
        lib.qa_device_supported.argtypes = [ctypes.c_int]
        lib.qa_device_supported.restype = ctypes.c_int
        vp = ctypes.c_void_p
        lib.qa_quantize_fp8.argtypes = [
            ctypes.c_int, ctypes.POINTER(vp), ctypes.c_int, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(vp),
            ctypes.POINTER(vp), vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.c_int,
            ctypes.c_int, vp,
        ]
        lib.qa_quantize_fp8.restype = ctypes.c_int
        lib.qa_quantize_workspace_floats.argtypes = [ctypes.c_int] * 4
        lib.qa_quantize_workspace_floats.restype = ctypes.c_size_t
        i64p = ctypes.POINTER(ctypes.c_int64)
        lib.qa_fp8_attn_fwd.argtypes = [
            vp, vp, vp, ctypes.c_int, i64p, i64p, i64p, vp, vp, vp, ctypes.c_int, vp, ctypes.c_int, vp,
            ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
            ctypes.c_float, ctypes.c_int, vp,
        ]
        lib.qa_fp8_attn_fwd.restype = ctypes.c_int
        lib.qa_fp8_attn_fwd_gated.argtypes = lib.qa_fp8_attn_fwd.argtypes[:-1] + [vp, ctypes.c_int, ctypes.c_int, vp]
        lib.qa_fp8_attn_fwd_gated.restype = ctypes.c_int
        lib.qa_set_flag.argtypes = [vp, vp]
        lib.qa_set_flag.restype = ctypes.c_int
        lib.qa_fp8_attn_func.argtypes = (
            [vp, vp, vp, ctypes.c_int, i64p, i64p, i64p, vp, vp, vp, vp, vp, vp, vp, ctypes.c_int, vp, vp]
            + [ctypes.c_int] * 7 + [ctypes.c_float, ctypes.c_int, ctypes.c_int, vp])
        lib.qa_fp8_attn_func.restype = ctypes.c_int
        lib.qa_attn_fwd.argtypes = ([vp, vp, vp, ctypes.c_int, i64p, i64p, i64p, vp, vp] + [ctypes.c_int] * 7
                                    + [ctypes.c_float, vp])
        lib.qa_attn_fwd.restype = ctypes.c_int
        lib.qa_merge_partials.argtypes = [vp, vp, vp, ctypes.c_int, vp, vp, ctypes.c_longlong, ctypes.c_int,
                                          ctypes.c_int, vp]
        lib.qa_merge_partials.restype = ctypes.c_int
        lib.qa_copy_2d.argtypes = [vp, ctypes.c_size_t, vp, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, vp]
        lib.qa_copy_2d.restype = ctypes.c_int
        szp = ctypes.POINTER(ctypes.c_size_t)
        lib.qa_copy_2d_batch.argtypes = [ctypes.c_int, ctypes.POINTER(vp), szp, ctypes.POINTER(vp), szp, szp, szp,
                                         ctypes.POINTER(vp)]
        lib.qa_copy_2d_batch.restype = ctypes.c_int
        if lib.qa_abi_version() != ABI_VERSION:
            raise NativeError(f"ABI mismatch: library {lib.qa_abi_version()} != binding {ABI_VERSION}")
        _lib = lib
    return _lib


def _check(rc: int, what: str):
    if rc != 0:
        msg = load().qa_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise NativeError(f"{what} failed (code {rc}): {msg}")


def _dt_code(dtype: torch.dtype) -> int:
    if dtype == torch.bfloat16:
        return QA_DT_BF16
    if dtype == torch.float16:
        return QA_DT_FP16
    if dtype == torch.float8_e4m3fn:
        return QA_DT_E4M3
    raise ValueError(f"unsupported dtype {dtype}")


def last_launch_count() -> int:
    return int(load().qa_last_launch_count())


_ws_floats = {}  # (B, H, S, D) -> qa_quantize_workspace_floats(...)
_ws_cache = {}  # (device index, raw stream handle) -> fp32 workspace, zero-filled when allocated, reused by every call
_I64x3 = ctypes.c_int64 * 3
_nullctx = contextlib.nullcontext()


def _dev_index(dev: torch.device) -> int:
    return dev.index if dev.index is not None else torch.cuda.current_device()


def _on_device(idx: int):
    """Device guard that costs nothing when ``idx`` already is the current device (the usual case)."""
    return _nullctx if torch.cuda.current_device() == idx else torch.cuda.device(idx)


def _raw_stream(idx: int) -> int:
    return torch._C._cuda_getCurrentRawStream(idx)


def _persistent_workspace(idx: int, n_floats: int) -> torch.Tensor:
    """The quantiser's workspace under the QA_WS_PERSISTENT contract of include/qattn.h: zeroed once, then only ever
    written by the library, one per (device, stream) so that the calls sharing it are stream-ordered.  Saves the
    per-call clear (a memset node and a dependency edge in front of every head-wise quantisation)."""
    key = (idx, _raw_stream(idx))
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < n_floats:
        with _on_device(idx):
            ws = torch.zeros((max(n_floats, 1 << 16),), dtype=torch.float32, device=torch.device("cuda", idx))
        _ws_cache[key] = ws
    return ws


def _workspace_for_call(idx: int, n_floats: int, workspace: Optional[torch.Tensor]):
    """-> (tensor, flags).  A caller-supplied workspace is plain scratch (cleared by the call).  While the stream is
    being captured into a CUDA graph the cached workspace is not used either: a fresh scratch tensor from the graph's
    own pool is cleared by a memset node of the graph, so replays neither depend on nor disturb state outside it.
    (The generation tag itself lives in device memory and advances per replay, so a C caller that does capture a
    persistent workspace is safe too.)"""
    dev = torch.device("cuda", idx)
    if workspace is not None:
        if workspace.dtype != torch.float32 or workspace.numel() < n_floats or workspace.device != dev:
            raise ValueError(f"quantize_fp8: workspace must be >= {n_floats} fp32 elements on {dev}")
        return workspace, 0
    if os.environ.get("QA_NO_PERSISTENT_WS") or torch.cuda.is_current_stream_capturing():
        return torch.empty((n_floats,), dtype=torch.float32, device=dev), 0
    return _persistent_workspace(idx, n_floats), QA_WS_PERSISTENT


def _in_place_ok(t: torch.Tensor) -> bool:
    """Whether the kernels can read ``t`` ([B,H,S,D]) through its own strides: D contiguous, 16-byte aligned rows."""
    if t.stride(3) != 1 or t.data_ptr() % 16:
        return False
    es = t.element_size()
    for size, st in zip(t.shape[:3], t.stride()[:3]):
        if size > 1 and (st <= 0 or (st * es) % 16):
            return False
    return t.stride(2) >= t.shape[3] or t.shape[2] == 1


def _strides4(t: torch.Tensor):
    """Element strides of a [B,H,S,D] tensor for the quantiser; size-1 dims take the dense value (frameworks report
    arbitrary strides there, and the library checks every stride for 16-byte alignment)."""
    B, H, S, D = t.shape
    dense = (H * S * D, S * D, D, 1)
    return [st if size > 1 else d for st, size, d in zip(t.stride(), t.shape, dense)]


def _strided(t: torch.Tensor):
    """-> (tensor the kernel reads, ctypes stride triple or None for a dense tensor)."""
    if t.is_contiguous():
        return t, None
    if not _in_place_ok(t):
        return t.contiguous(), None
    return t, _I64x3(*t.stride()[:3])


def quantize_fp8(tensors: Sequence[torch.Tensor], scale_mode: int,
                 scales: Optional[Sequence[torch.Tensor]] = None,
                 workspace: Optional[torch.Tensor] = None,
                 outs: Optional[Sequence[torch.Tensor]] = None) -> Tuple[list, list]:
    """Quantise 1-3 CUDA tensors [B,H,S_i,D] (bf16/fp16, same B,H,D,dtype) in one launch pair.

    Returns ([e4m3 tensors], [fp32 scales: [B,H] head-wise or [B,H,S_i] token-wise]).
    ``workspace``: optional caller-owned scratch (plain contract: contents ignored); by default a per-(device, stream)
    workspace under the QA_WS_PERSISTENT contract is used, which saves the per-call clear.
    ``QA_SCALE_HEAD_AMAX_ONLY`` returns ([], scales) without quantising; ``QA_SCALE_HEAD_GIVEN`` quantises with the
    fp32 [B,H] ``scales`` passed in.  ``outs``: optional dense e4m3 / uint8 destinations of the inputs' shapes (e.g.
    views of a peer-visible communication buffer).
    """
    lib = load()
    n = len(tensors)
    t0 = tensors[0]
    B, H, _, D = t0.shape
    dev = t0.device
    idx = _dev_index(dev)
    xs = []
    for t in tensors:
        if t.device != dev or t.dtype != t0.dtype or t.dim() != 4 or t.shape[0] != B or t.shape[1] != H or t.shape[3] != D:
            raise ValueError("quantize_fp8: tensors must share device, dtype, B, H and D")
        if not t.is_contiguous() and not _in_place_ok(t):
            t = t.contiguous()
        xs.append(t)
    amax_only = scale_mode == QA_SCALE_HEAD_AMAX_ONLY
    with _on_device(idx):
        if amax_only:
            outs = []
        elif outs is None:
            outs = [torch.empty(t.shape, dtype=torch.float8_e4m3fn, device=dev) for t in xs]
        else:
            outs = list(outs)
            if len(outs) != n or any(o.shape != t.shape or o.element_size() != 1 or not o.is_contiguous() or o.device != dev
                                     for o, t in zip(outs, xs)):
                raise ValueError("quantize_fp8: `outs` must be dense 1-byte tensors of the inputs' shapes and device")
        if scale_mode == QA_SCALE_HEAD_GIVEN:
            if scales is None or len(scales) != n:
                raise ValueError("quantize_fp8: QA_SCALE_HEAD_GIVEN needs one [B,H] fp32 scale tensor per input")
            scales = [s_.to(device=dev, dtype=torch.float32).reshape(B, H).contiguous() for s_ in scales]
            ws, ws_ptr = None, None
        elif scale_mode in (QA_SCALE_HEAD, QA_SCALE_HEAD_TWO_PASS, QA_SCALE_HEAD_AMAX_ONLY, QA_SCALE_HEAD_RELOAD):
            scales = [torch.empty((B, H), dtype=torch.float32, device=dev) for _ in xs]
            n_ws = int(lib.qa_quantize_workspace_floats(B, H, max(t.shape[2] for t in xs), D))
            ws, flags = _workspace_for_call(idx, n_ws, workspace)
            scale_mode |= flags
            ws_ptr = ws.data_ptr()
        else:
            scales = [torch.empty((B, H, t.shape[2]), dtype=torch.float32, device=dev) for t in xs]
            ws, ws_ptr = None, None
        vp = ctypes.c_void_p
        x_arr = (vp * n)(*[t.data_ptr() for t in xs])
        o_arr = (vp * n)(*[t.data_ptr() for t in outs]) if outs else (vp * n)()
        s_arr = (vp * n)(*[t.data_ptr() for t in scales])
        strides = (ctypes.c_int64 * (4 * n))(*[s for t in xs for s in _strides4(t)])
        S = (ctypes.c_int * n)(*[t.shape[2] for t in xs])
        stream = _raw_stream(idx)
        if quant_events is not None:
            tstream = torch.cuda.current_stream(dev)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(tstream)
        rc = lib.qa_quantize_fp8(n, x_arr, _dt_code(t0.dtype), strides, o_arr, s_arr, ws_ptr, B, H, S, D,
                                 scale_mode, stream)
        if quant_events is not None:
            ev1.record(tstream)
            quant_events.append((ev0, ev1))
    _check(rc, "qa_quantize_fp8")
    global launch_total
    launch_total += int(lib.qa_last_launch_count())
    return outs, scales


def _f32c(t: Optional[torch.Tensor]):
    if t is None or (t.dtype == torch.float32 and t.is_contiguous()):
        return t
    return t.to(torch.float32).contiguous()


def fp8_attn_fwd(q8: torch.Tensor, k8: torch.Tensor, v: torch.Tensor, scale_q: torch.Tensor, scale_k: torch.Tensor,
                 scale_v: Optional[torch.Tensor], *, scale_mode: int, is_causal, sm_scale: float, p_mode: int,
                 out_dtype: torch.dtype, return_lse: bool = False, out: Optional[torch.Tensor] = None, gate=None):
    """Launch the fused forward kernel.  q8/k8 e4m3 [B,H,S,D]; v e4m3 (+scale_v) or bf16/fp16.  Tensors whose last
    dim is contiguous and whose strides are 16-byte multiples ([B,S,H,D]-held views) are read in place.  ``is_causal``:
    a bool (top-left mask) or QA_CAUSAL_BOTTOM_RIGHT (row i sees keys <= i + Skv - Sq; Sq <= Skv).  ``out``:
    optional dense [B,Hq,Sq,D] destination (e.g. a head range of a larger output).  ``gate``: optional
    (flags int32 tensor, heads_per_gate, flags_per_gate) - a gated launch (``qa_fp8_attn_fwd_gated``): the CTAs of kv
    head h read K / V only once flags[(h // heads_per_gate) * flags_per_gate : ... + flags_per_gate] are non-zero
    (``set_flag`` on the streams that bring them)."""
    lib = load()
    B, Hq, Sq, D = q8.shape
    Hkv, Skv = k8.shape[1], k8.shape[2]
    dev = q8.device
    idx = _dev_index(dev)
    if scale_q.numel() != (B * Hq if scale_mode == QA_SCALE_HEAD else B * Hq * Sq) or \
            scale_k.numel() != (B * Hkv if scale_mode == QA_SCALE_HEAD else B * Hkv * Skv):
        raise ValueError(f"scale_q / scale_k have {scale_q.numel()} / {scale_k.numel()} elements, which does not match "
                         f"{'head-wise [B,H]' if scale_mode == QA_SCALE_HEAD else 'token-wise [B,H,S]'} scales")
    if scale_v is not None and scale_v.numel() != B * Hkv:
        raise ValueError(f"scale_v must have B*Hkv = {B * Hkv} elements")
    (q8, qs), (k8, ks), (v, vs) = _strided(q8), _strided(k8), _strided(v)
    scale_q, scale_k, scale_v = _f32c(scale_q), _f32c(scale_k), _f32c(scale_v)
    if out is not None and (out.shape != (B, Hq, Sq, D) or out.dtype != out_dtype or not out.is_contiguous()
                            or out.device != dev):
        raise ValueError("fp8_attn_fwd: `out` must be a dense [B,Hq,Sq,D] tensor of out_dtype on the inputs' device")
    with _on_device(idx):
        if out is None:
            out = torch.empty((B, Hq, Sq, D), dtype=out_dtype, device=dev)
        lse = torch.empty((B, Hq, Sq), dtype=torch.float32, device=dev) if return_lse else None
        stream = _raw_stream(idx)
        if attn_events is not None:
            tstream = torch.cuda.current_stream(dev)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(tstream)
        common = (q8.data_ptr(), k8.data_ptr(), v.data_ptr(), _dt_code(v.dtype), qs, ks, vs, scale_q.data_ptr(),
                  scale_k.data_ptr(), scale_v.data_ptr() if scale_v is not None else None, scale_mode, out.data_ptr(),
                  _dt_code(out_dtype), lse.data_ptr() if lse is not None else None, B, Hq, Hkv, Sq, Skv, D,
                  int(is_causal), float(sm_scale), p_mode)
        if gate is None:
            rc = lib.qa_fp8_attn_fwd(*common, stream)
        else:
            flags, heads_per_gate, flags_per_gate = gate
            n_gates = -(-Hkv // int(heads_per_gate))
            if flags.dtype != torch.int32 or flags.device != dev or not flags.is_contiguous() or \
                    flags.numel() < n_gates * int(flags_per_gate):
                raise ValueError("fp8_attn_fwd: `gate` needs a dense int32 flag tensor on the inputs' device with "
                                 "ceil(Hkv / heads_per_gate) * flags_per_gate words")
            rc = lib.qa_fp8_attn_fwd_gated(*common, flags.data_ptr(), int(heads_per_gate), int(flags_per_gate), stream)
        if attn_events is not None:
            ev1.record(tstream)
            attn_events.append((ev0, ev1))
    _check(rc, "qa_fp8_attn_fwd")
    global launch_total
    launch_total += int(lib.qa_last_launch_count())
    return (out, lse) if return_lse else out


def _align(n: int, a: int = 256) -> int:
    return (n + a - 1) // a * a


def fp8_attn_func(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, scale_mode: int, is_causal: bool,
                  sm_scale: float, p_mode: int, return_lse: bool = False, return_quantized: bool = False):
    """16-bit q, k, v -> attention output in ONE crossing of the C ABI (``qa_fp8_attn_func``: quantise + fused forward).

    All intermediates (e4m3 tensors and scales) live in one scratch allocation.  With ``return_quantized`` the call also
    returns ``dict(q8, k8, v8, scale_q, scale_k, scale_v)`` (views of that scratch) so K / V can be reused by later
    ``fp8_attn_fwd`` calls."""
    lib = load()
    B, Hq, Sq, D = q.shape
    Hkv, Skv = k.shape[1], k.shape[2]
    dev = q.device
    idx = _dev_index(dev)
    token = scale_mode == QA_SCALE_TOKEN
    v_fp8 = p_mode != QA_P_16BIT
    (q, qs), (k, ks), (v, vs) = _strided(q), _strided(k), _strided(v)
    nq, nk = B * Hq * Sq * D, B * Hkv * Skv * D
    nsq, nsk, nsv = (B * Hq * Sq, B * Hkv * Skv, B * Hkv) if token else (B * Hq, B * Hkv, B * Hkv)
    o_k8 = _align(nq)
    o_v8 = o_k8 + _align(nk)
    o_sq = o_v8 + (_align(nk) if v_fp8 else 0)
    o_sk = o_sq + _align(4 * nsq)
    o_sv = o_sk + _align(4 * nsk)
    total = o_sv + _align(4 * nsv)
    with _on_device(idx):
        buf = torch.empty((total,), dtype=torch.uint8, device=dev)
        out = torch.empty((B, Hq, Sq, D), dtype=q.dtype, device=dev)
        lse = torch.empty((B, Hq, Sq), dtype=torch.float32, device=dev) if return_lse else None
        ws_ptr, flags = None, 0
        if not token or v_fp8:
            wkey = (B, max(Hq, Hkv), max(Sq, Skv), D)
            n_ws = _ws_floats.get(wkey)
            if n_ws is None:
                n_ws = _ws_floats[wkey] = int(lib.qa_quantize_workspace_floats(*wkey))
            ws, flags = _workspace_for_call(idx, n_ws, None)
            ws_ptr = ws.data_ptr()
        base = buf.data_ptr()
        rc = lib.qa_fp8_attn_func(
            q.data_ptr(), k.data_ptr(), v.data_ptr(), _dt_code(q.dtype), qs, ks, vs, base, base + o_k8,
            (base + o_v8) if v_fp8 else None, base + o_sq, base + o_sk, (base + o_sv) if v_fp8 else None, ws_ptr, flags,
            out.data_ptr(), lse.data_ptr() if lse is not None else None, B, Hq, Hkv, Sq, Skv, D, int(bool(is_causal)),
            float(sm_scale), scale_mode, p_mode, _raw_stream(idx),
        )
    _check(rc, "qa_fp8_attn_func")
    global launch_total
    launch_total += int(lib.qa_last_launch_count())
    res = (out, lse) if return_lse else out
    if not return_quantized:
        return res
    f8, f32 = torch.float8_e4m3fn, torch.float32
    sq_shape, sk_shape = ((B, Hq, Sq), (B, Hkv, Skv)) if token else ((B, Hq), (B, Hkv))
    quant = {
        "q8": buf[:nq].view(f8).view(B, Hq, Sq, D), "k8": buf[o_k8:o_k8 + nk].view(f8).view(B, Hkv, Skv, D),
        "v8": buf[o_v8:o_v8 + nk].view(f8).view(B, Hkv, Skv, D) if v_fp8 else None,
        "scale_q": buf[o_sq:o_sq + 4 * nsq].view(f32).view(sq_shape),
        "scale_k": buf[o_sk:o_sk + 4 * nsk].view(f32).view(sk_shape),
        "scale_v": buf[o_sv:o_sv + 4 * nsv].view(f32).view(B, Hkv) if v_fp8 else None,
    }
    return res, quant


def attn_fwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, is_causal, sm_scale: float,
             return_lse: bool = False):
    """Launch the fused forward kernel on 16-bit q, k, v (all bf16 or all fp16), [B,H,S,D] (strided views are read in
    place when their strides are 16-byte multiples).  ``is_causal`` as in ``fp8_attn_fwd``."""
    lib = load()
    B, Hq, Sq, D = q.shape
    Hkv, Skv = k.shape[1], k.shape[2]
    dev = q.device
    idx = _dev_index(dev)
    (q, qs), (k, ks), (v, vs) = _strided(q), _strided(k), _strided(v)
    with _on_device(idx):
        out = torch.empty((B, Hq, Sq, D), dtype=q.dtype, device=dev)
        lse = torch.empty((B, Hq, Sq), dtype=torch.float32, device=dev) if return_lse else None
        if attn_events is not None:
            tstream = torch.cuda.current_stream(dev)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(tstream)
        rc = lib.qa_attn_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), _dt_code(q.dtype), qs, ks, vs, out.data_ptr(),
                             lse.data_ptr() if lse is not None else None, B, Hq, Hkv, Sq, Skv, D,
                             int(is_causal), float(sm_scale), _raw_stream(idx))
        if attn_events is not None:
            ev1.record(tstream)
            attn_events.append((ev0, ev1))
    _check(rc, "qa_attn_fwd")
    global launch_total
    launch_total += int(lib.qa_last_launch_count())
    return (out, lse) if return_lse else out


def merge_partials(o_acc: Optional[torch.Tensor], lse_acc: torch.Tensor, o_new: torch.Tensor, lse_new: torch.Tensor,
                   *, first: bool, out: Optional[torch.Tensor] = None) -> None:
    """(o_acc, lse_acc) <- combine with the partial result (o_new, lse_new) of one key block (include/qattn.h).

    o_acc fp32 [..., D] / lse_acc fp32 [...]; o_new 16-bit, lse_new fp32.  With ``out`` (16-bit) the merged rows go
    there instead of into o_acc (the last ring step)."""
    lib = load()
    D = o_new.shape[-1]
    rows = o_new.numel() // D
    for t in (o_acc, lse_acc, o_new, lse_new, out):
        if t is not None and not t.is_contiguous():
            raise ValueError("merge_partials: tensors must be contiguous")
    if lse_acc.dtype != torch.float32 or lse_new.dtype != torch.float32 or (o_acc is not None and o_acc.dtype != torch.float32):
        raise ValueError("merge_partials: accumulators and LSE must be fp32")
    idx = _dev_index(o_new.device)
    with _on_device(idx):
        stream = _raw_stream(idx)
        rc = lib.qa_merge_partials(o_acc.data_ptr() if o_acc is not None else None, lse_acc.data_ptr(),
                                   o_new.data_ptr(), _dt_code(o_new.dtype), lse_new.data_ptr(),
                                   out.data_ptr() if out is not None else None, rows, D, int(bool(first)), stream)
    _check(rc, "qa_merge_partials")
    global launch_total
    launch_total += int(lib.qa_last_launch_count())


def copy_2d(dst_ptr: int, dst_pitch: int, src_ptr: int, src_pitch: int, width_bytes: int, rows: int, stream: int) -> None:
    """Asynchronous strided block copy on the copy engines (``qa_copy_2d``); raw device addresses and a raw stream."""
    _check(load().qa_copy_2d(dst_ptr, dst_pitch, src_ptr, src_pitch, width_bytes, rows, stream), "qa_copy_2d")


def set_flag(flags: torch.Tensor, index: int, raw_stream: int) -> None:
    """flags[index] = non-zero in the order of ``raw_stream`` (``qa_set_flag``: a stream memory operation behind the
    copies it vouches for - no kernel, so it completes even while a polling launch holds every SM)."""
    _check(load().qa_set_flag(flags.data_ptr() + 4 * int(index), raw_stream), "qa_set_flag")


class CopyBatch:
    """A fixed list of strided block copies (``qa_copy_2d_batch``) marshalled once and issued with one call."""

    def __init__(self, copies):
        """copies: sequence of (dst_ptr, dst_pitch, src_ptr, src_pitch, width_bytes, rows, raw_stream)."""
        n = self.n = len(copies)
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        cols = list(zip(*copies)) if n else [[]] * 7
        self.args = ((vp * n)(*cols[0]), (sz * n)(*cols[1]), (vp * n)(*cols[2]), (sz * n)(*cols[3]), (sz * n)(*cols[4]),
                     (sz * n)(*cols[5]), (vp * n)(*cols[6]))

    def issue(self) -> None:
        a = self.args
        _check(load().qa_copy_2d_batch(self.n, a[0], a[1], a[2], a[3], a[4], a[5], a[6]), "qa_copy_2d_batch")
