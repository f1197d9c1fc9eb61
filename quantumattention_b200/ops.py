"""torch custom ops of the hot path, same names and schemas as the reference so traced graphs look the same
(reference: src/quantum_attn/ops.py:32-147):

    quantum_attn::fp8_attention_forward(query, key, value, scale_q, scale_k, attn_mask, dropout_p, is_causal, *, scale)
    quantum_attn::attention_forward(query, key, value, attn_mask, dropout_p, is_causal, *, scale)

plus two ops the reference does not need because its quantiser is traced into aten ops and compiled by Inductor
(src/quantum_attn/nn.py:14-42) - here the quantiser is a hand-written kernel, and a traced graph must call IT:

    quantum_attn::dynamically_quantize_fp8(t, reduction_dim) -> (t_fp8, scale)
    quantum_attn::quantize_qk_fp8(query, key, token_wise) -> (q_fp8, k_fp8, scale_q, scale_k)     (one launch)

The CUDA implementation calls the sm_100a kernels through the C ABI (``_native``); the reference's CUDA implementation
is aten SDPA on the dequantised inputs, which survives here only as ``fp8_attention_definition`` - the semantic
definition used for fake-tensor shape inference and as an explicit debug comparator.
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import torch

from . import _native, config

aten = torch.ops.aten

_PV_MODES = {"fp8": _native.QA_P_E4M3, "fp8_hilo": _native.QA_P_E4M3_HILO, "16bit": _native.QA_P_16BIT}


def pv_mode_code(name: Optional[str] = None) -> int:
    name = config.attention.pv_mode if name is None else name
    try:
        return _PV_MODES[name]
    except KeyError:
        raise ValueError(f"Unsupported pv_mode: {name} (expected one of {sorted(_PV_MODES)})") from None


def fp8_attention_definition(query, key, value, scale_q=None, scale_k=None, attn_mask=None, dropout_p=0.0,
                             is_causal=False, *, scale=None):
    """What the op computes, stated with aten ops (reference: src/quantum_attn/ops.py:64-95)."""
    out_dtype = value.dtype
    query = query.to(out_dtype)
    key = key.to(out_dtype)
    if scale_q is not None:
        sq, sk = scale_q.to(out_dtype), scale_k.to(out_dtype)
        while sq.dim() < query.dim():
            sq, sk = sq.unsqueeze(-1), sk.unsqueeze(-1)
        query, key = query * sq, key * sk
    if key.size(1) != query.size(1):  # GQA (extension; the reference's Python gate forbids it)
        rep = query.size(1) // key.size(1)
        key, value = key.repeat_interleave(rep, 1), value.repeat_interleave(rep, 1)
    return aten.scaled_dot_product_attention(
        query, key, value, attn_mask=attn_mask, dropout_p=dropout_p, is_causal=is_causal, scale=scale
    ).contiguous()


def attention_definition(query, key, value, attn_mask=None, dropout_p=0.0, is_causal=False, *, scale=None):
    """What the 16-bit op computes, stated with aten ops (reference: src/quantum_attn/ops.py:27-29)."""
    if key.size(1) != query.size(1):  # GQA (extension; the reference's Python gate forbids it)
        rep = query.size(1) // key.size(1)
        key, value = key.repeat_interleave(rep, 1), value.repeat_interleave(rep, 1)
    return aten.scaled_dot_product_attention(
        query, key, value, attn_mask=attn_mask, dropout_p=dropout_p, is_causal=is_causal, scale=scale
    ).contiguous()


def attention_native(query, key, value, is_causal=False, scale=None, return_lse=False):
    """16-bit q, k, v -> attention output through the sm_100a kernel (no fallback)."""
    if query.dtype not in (torch.float16, torch.bfloat16) or key.dtype != query.dtype or value.dtype != query.dtype:
        raise ValueError("attention_forward expects query, key and value of one dtype, torch.float16 or torch.bfloat16")
    sm_scale = (1.0 / math.sqrt(query.size(-1))) if scale is None else float(scale)
    return _native.attn_fwd(query, key, value, is_causal=bool(is_causal), sm_scale=sm_scale, return_lse=return_lse)


def _scale_mode_of(scale_q: torch.Tensor, query: torch.Tensor, scale_k: Optional[torch.Tensor] = None,
                   key: Optional[torch.Tensor] = None) -> int:
    """Granularity of the scales, from their RANK as in the reference (src/quantum_attn/ops.py:76-83 broadcasts a
    rank-(n-2) or rank-(n-1) scale over the tensor), with the shapes checked against the tensors they scale - the
    kernel indexes scale_q[B*H(*S)] and scale_k[B*Hkv(*Skv)] without looking at their extents."""
    def one(s, t, name):
        if s.dim() == t.dim() - 2 and tuple(s.shape) == tuple(t.shape[:-2]):
            return _native.QA_SCALE_HEAD
        if s.dim() == t.dim() - 1 and tuple(s.shape) == tuple(t.shape[:-1]):
            return _native.QA_SCALE_TOKEN
        raise ValueError(f"{name} of shape {tuple(s.shape)} matches neither the head-wise shape {tuple(t.shape[:-2])} "
                         f"nor the token-wise shape {tuple(t.shape[:-1])} of its tensor")
    mode = one(scale_q, query, "scale_q")
    if scale_k is not None and one(scale_k, key, "scale_k") != mode:
        raise ValueError("scale_q and scale_k must have the same granularity (both head-wise or both token-wise)")
    return mode


def fp8_attention_native(query, key, value, scale_q, scale_k, is_causal=False, scale=None, pv_mode=None,
                         return_lse=False, scale_v=None, out_dtype=None):
    """q8/k8 (e4m3) + scales + V -> attention output through the sm_100a kernels (no fallback).

    V is 16-bit (quantised here in the FP8 P modes) or - with ``scale_v`` - already e4m3 with head-wise scales (the
    K8 / V8 reuse path: quantise K and V once, attend many times)."""
    if query.dtype != torch.float8_e4m3fn or key.dtype != torch.float8_e4m3fn:
        raise ValueError("fp8_attention_forward expects float8_e4m3fn query and key")
    if scale_q is None or scale_k is None:
        raise ValueError("fp8_attention_forward needs scale_q and scale_k")
    mode = pv_mode_code(pv_mode)
    scale_mode = _scale_mode_of(scale_q, query, scale_k, key)
    sm_scale = (1.0 / math.sqrt(query.size(-1))) if scale is None else float(scale)
    if value.dtype == torch.float8_e4m3fn:
        if scale_v is None:
            raise ValueError("an e4m3 value tensor needs its head-wise scale_v")
        if mode == _native.QA_P_16BIT:
            raise ValueError("an e4m3 value tensor needs pv_mode 'fp8' or 'fp8_hilo' (the '16bit' mode multiplies the "
                             "16-bit value tensor)")
        v_in = value
    elif scale_v is not None:
        raise ValueError("scale_v goes with a float8_e4m3fn value tensor")
    elif mode == _native.QA_P_16BIT:
        v_in = value
    else:
        (v_in,), (scale_v,) = _native.quantize_fp8([value], _native.QA_SCALE_HEAD)
    if out_dtype is None:
        out_dtype = value.dtype if value.dtype in (torch.float16, torch.bfloat16) else torch.bfloat16
    return _native.fp8_attn_fwd(query, key, v_in, scale_q, scale_k, scale_v, scale_mode=scale_mode,
                                is_causal=bool(is_causal), sm_scale=sm_scale, p_mode=mode, out_dtype=out_dtype,
                                return_lse=return_lse)


@torch.library.custom_op("quantum_attn::fp8_attention_forward", mutates_args=(), device_types=("cuda",))
def fp8_attention_forward(
    query: torch.Tensor,
    key: torch.Tensor,
    value: torch.Tensor,
    scale_q: Optional[torch.Tensor] = None,
    scale_k: Optional[torch.Tensor] = None,
    attn_mask: Optional[torch.Tensor] = None,
    dropout_p: float = 0.0,
    is_causal: bool = False,
    *,
    scale: Optional[float] = None,
) -> torch.Tensor:
    if attn_mask is not None or dropout_p != 0.0:
        raise ValueError("NYI: attn_mask must be None and dropout_p must be 0.0")
    if config.attention.force_eager_fallback:
        return fp8_attention_definition(query, key, value, scale_q, scale_k, attn_mask, dropout_p, is_causal,
                                        scale=scale)
    return fp8_attention_native(query, key, value, scale_q, scale_k, is_causal=is_causal, scale=scale)


@torch.library.register_fake("quantum_attn::fp8_attention_forward")
def _(query, key, value, scale_q=None, scale_k=None, attn_mask=None, dropout_p=0.0, is_causal=False, *, scale=None):
    return torch.empty(query.shape[:-1] + (value.shape[-1],), dtype=value.dtype, device=query.device)


@torch.library.custom_op("quantum_attn::attention_forward", mutates_args=(), device_types=("cuda",))
def attention_forward(
    query: torch.Tensor,
    key: torch.Tensor,
    value: torch.Tensor,
    attn_mask: Optional[torch.Tensor] = None,
    dropout_p: float = 0.0,
    is_causal: bool = False,
    *,
    scale: Optional[float] = None,
) -> torch.Tensor:
    # 16-bit QK^T path (reference: src/quantum_attn/ops.py:32-45): the same fused kernel with kind::f16 MMAs
    if attn_mask is not None or dropout_p != 0.0:
        raise ValueError("NYI: attn_mask must be None and dropout_p must be 0.0")
    if config.attention.force_eager_fallback:
        return attention_definition(query, key, value, attn_mask, dropout_p, is_causal, scale=scale)
    return attention_native(query, key, value, is_causal=is_causal, scale=scale)


@torch.library.register_fake("quantum_attn::attention_forward")
def _(query, key, value, attn_mask=None, dropout_p=0.0, is_causal=False, *, scale=None):
    return torch.empty(query.shape[:-1] + (value.shape[-1],), dtype=value.dtype, device=query.device)


# ------------------------------------------------------------------------------------------------ quantiser ops
def _norm_dims(reduction_dim, ndim):
    dims = list(reduction_dim) if isinstance(reduction_dim, (list, tuple)) else [reduction_dim]
    return sorted(int(d) % ndim for d in dims)


def quantize_native(t: torch.Tensor, reduction_dim):
    """The hand-written quantiser on one tensor: reduce over the last dim (token-wise) or the last two (head-wise)."""
    dims = _norm_dims(reduction_dim, t.dim())
    if t.device.type != "cuda":
        raise ValueError("Expected the tensor to be on a CUDA device")
    if t.dtype not in (torch.float16, torch.bfloat16):
        raise ValueError(f"Expected dtype torch.float16 or torch.bfloat16, but got {t.dtype} instead.")
    if t.dim() < 2 or t.size(-1) not in (64, 128, 256):
        raise ValueError(f"Unsupported head dimension: {t.size(-1) if t.dim() else None}")
    if dims == [t.dim() - 1]:
        mode, lead = _native.QA_SCALE_TOKEN, t.shape[:-1]
        x = t.reshape(1, 1, -1, t.size(-1))
    elif dims == [t.dim() - 2, t.dim() - 1]:
        mode, lead = _native.QA_SCALE_HEAD, t.shape[:-2]
        x = t.reshape(1, -1, t.size(-2), t.size(-1)) if t.dim() != 4 else t
    else:
        raise ValueError(f"Unsupported reduction_dim: {reduction_dim}")
    (x8,), (scale,) = _native.quantize_fp8([x], mode)
    return x8.reshape(t.shape), scale.reshape(lead)


@torch.library.custom_op("quantum_attn::dynamically_quantize_fp8", mutates_args=(), device_types=("cuda",))
def dynamically_quantize_fp8_op(t: torch.Tensor, reduction_dim: List[int]) -> Tuple[torch.Tensor, torch.Tensor]:
    # what a traced `dynamically_quantize_fp8` resolves to: the sm_100a quantise kernel, not Inductor-generated code
    return quantize_native(t, reduction_dim)


@torch.library.register_fake("quantum_attn::dynamically_quantize_fp8")
def _(t, reduction_dim):
    dims = _norm_dims(reduction_dim, t.dim())
    lead = [s for i, s in enumerate(t.shape) if i not in dims]
    return (torch.empty(t.shape, dtype=torch.float8_e4m3fn, device=t.device),
            torch.empty(lead, dtype=torch.float32, device=t.device))


def quantize_qk_native(query: torch.Tensor, key: torch.Tensor, token_wise: bool):
    mode = _native.QA_SCALE_TOKEN if token_wise else _native.QA_SCALE_HEAD
    if query.shape[1] == key.shape[1]:
        (q8, k8), (sq, sk) = _native.quantize_fp8([query, key], mode)  # one launch for both
    else:
        (q8,), (sq,) = _native.quantize_fp8([query], mode)
        (k8,), (sk,) = _native.quantize_fp8([key], mode)
    return q8, k8, sq, sk


@torch.library.custom_op("quantum_attn::quantize_qk_fp8", mutates_args=(), device_types=("cuda",))
def quantize_qk_fp8_op(query: torch.Tensor, key: torch.Tensor, token_wise: bool
                       ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    # the Q / K quantisation of `_fp8_attention_wrapper` (reference: src/quantum_attn/nn.py:410-418) as ONE launch
    return quantize_qk_native(query, key, token_wise)


@torch.library.register_fake("quantum_attn::quantize_qk_fp8")
def _(query, key, token_wise):
    cut = -1 if token_wise else -2
    return (torch.empty(query.shape, dtype=torch.float8_e4m3fn, device=query.device),
            torch.empty(key.shape, dtype=torch.float8_e4m3fn, device=key.device),
            torch.empty(query.shape[:cut], dtype=torch.float32, device=query.device),
            torch.empty(key.shape[:cut], dtype=torch.float32, device=key.device))
