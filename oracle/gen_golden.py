"""Generate tests/golden/*.npz by running the REFERENCE's own pure-torch pieces on CPU in the build container.

Run once, with a checkout of the reference (never at test time):
    python oracle/gen_golden.py <reference checkout>/src

What is recorded
  * quantize_{head,token}.npz - inputs (bf16 bit patterns) and the outputs of the reference's
    ``quantum_attn.nn._dynamically_quantize_fp8`` (src/quantum_attn/nn.py:14-19) applied to the fp32-widened input
    with the reduction dims of src/quantum_attn/nn.py:410-418.  fp32 intermediates are what the reference's default
    (Inductor-fused) path computes.  The eager-bf16 outputs are stored too (``*_eager_bf16``) for information.
  * attn_*.npz - q8/k8 bytes, scales, v, and the output of ``quantum_attn.ops._fp8_attention_forward``
    (src/quantum_attn/ops.py:64-95) on CPU, in bf16 (the reference's arithmetic) and with fp32 tensors.

The reference does not import on torch 2.11 without a one-line shim (SURVEY.md §8c): ``use_max_autotune`` was
removed from torch._inductor.utils; the shim only affects the Inductor lowering module, which is not exercised.
"""
import os
import sys

import numpy as np
import torch

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def import_reference(ref_src):
    import torch._inductor.utils as iu

    if not hasattr(iu, "use_max_autotune"):
        iu.use_max_autotune = lambda: False
    sys.path.insert(0, ref_src)
    import quantum_attn  # noqa: F401
    from quantum_attn import nn as ref_nn, ops as ref_ops

    return ref_nn, ref_ops


def bf16_bits(t):
    return t.contiguous().view(torch.int16).numpy().copy()


def main(ref_src):
    ref_nn, ref_ops = import_reference(ref_src)
    os.makedirs(OUT, exist_ok=True)
    g = torch.Generator(device="cpu").manual_seed(1234)

    # ---- quantiser vectors
    for mode, dims in (("head", [2, 3]), ("token", 3)):
        x = torch.randn(2, 3, 77, 64, generator=g) * torch.exp(torch.randn(2, 3, 1, 64, generator=g))
        x[0, 1] = 0  # all-zero head: scale clamps to eps
        x[1, 2, 5, 7] = 3.0e4  # large outlier
        x = x.to(torch.bfloat16)
        y32, s32 = ref_nn._dynamically_quantize_fp8(x.float(), reduction_dim=dims)
        ybf, sbf = ref_nn._dynamically_quantize_fp8(x, reduction_dim=dims)
        np.savez_compressed(
            os.path.join(OUT, f"quantize_{mode}.npz"),
            x_bf16_bits=bf16_bits(x),
            q_bytes=y32.view(torch.uint8).numpy(),
            scale=s32.numpy(),
            q_bytes_eager_bf16=ybf.view(torch.uint8).numpy(),
            scale_eager_bf16=sbf.numpy(),
        )

    # ---- attention vectors (small shapes, both causal settings, ragged S)
    for name, (B, H, Sq, Skv, D, causal, mode) in {
        "attn_d64_causal": (1, 2, 200, 200, 64, True, "head"),
        "attn_d128": (1, 2, 130, 257, 128, False, "head"),
        "attn_d128_token": (1, 2, 96, 160, 128, False, "token"),
        "attn_d256_causal": (1, 1, 160, 160, 256, True, "head"),
    }.items():
        q = torch.randn(B, H, Sq, D, generator=g).to(torch.bfloat16)
        k = torch.randn(B, H, Skv, D, generator=g).to(torch.bfloat16)
        v = torch.randn(B, H, Skv, D, generator=g).to(torch.bfloat16)
        dims = [2, 3] if mode == "head" else 3
        q8, sq = ref_nn._dynamically_quantize_fp8(q.float(), reduction_dim=dims)
        k8, sk = ref_nn._dynamically_quantize_fp8(k.float(), reduction_dim=dims)
        out_bf16 = ref_ops._fp8_attention_forward(q8, k8, v, sq, sk, is_causal=causal)
        out_fp32 = ref_ops._fp8_attention_forward(q8, k8, v.float(), sq, sk, is_causal=causal)
        np.savez_compressed(
            os.path.join(OUT, f"{name}.npz"),
            q8=q8.view(torch.uint8).numpy(),
            k8=k8.view(torch.uint8).numpy(),
            scale_q=sq.numpy(),
            scale_k=sk.numpy(),
            v_bf16_bits=bf16_bits(v),
            q_bf16_bits=bf16_bits(q),
            k_bf16_bits=bf16_bits(k),
            out_ref_bf16_bits=bf16_bits(out_bf16),
            out_ref_fp32=out_fp32.numpy(),
            causal=np.array(causal),
        )
    # ---- 16-bit attention vectors: the reference's `_attention_forward` (src/quantum_attn/ops.py:15-28) on CPU, in the
    # input dtype (its arithmetic) and on the fp32-widened tensors.  Own generator: the files above stay byte-identical.
    g16 = torch.Generator(device="cpu").manual_seed(4321)
    for name, (B, Hq, Hkv, Sq, Skv, D, causal, dtype) in {
        "attn16_d64_causal": (1, 2, 2, 200, 200, 64, True, torch.bfloat16),
        "attn16_d128": (1, 2, 2, 130, 257, 128, False, torch.bfloat16),
        "attn16_d128_fp16_causal": (2, 2, 2, 300, 300, 128, True, torch.float16),
        "attn16_d256_causal": (1, 1, 1, 160, 160, 256, True, torch.bfloat16),
    }.items():
        q = torch.randn(B, Hq, Sq, D, generator=g16).to(dtype)
        k = torch.randn(B, Hkv, Skv, D, generator=g16).to(dtype)
        v = torch.randn(B, Hkv, Skv, D, generator=g16).to(dtype)
        out_16 = ref_ops._attention_forward(q, k, v, is_causal=causal)
        out_fp32 = ref_ops._attention_forward(q.float(), k.float(), v.float(), is_causal=causal)
        # heads are independent: the B = 2 fixture keeps head 0 of each batch element, so that its file stays under 1 MB
        h = 1 if name == "attn16_d128_fp16_causal" else Hq
        q, k, v, out_16, out_fp32 = (t[:, :h] for t in (q, k, v, out_16, out_fp32))
        np.savez_compressed(
            os.path.join(OUT, f"{name}.npz"),
            q_bits=bf16_bits(q), k_bits=bf16_bits(k), v_bits=bf16_bits(v),  # int16 views (bf16 or fp16 bit patterns)
            fp16=np.array(dtype == torch.float16),
            out_ref_16_bits=bf16_bits(out_16),
            out_ref_fp32=out_fp32.numpy(),
            causal=np.array(causal),
        )
    print("golden vectors written to", os.path.normpath(OUT))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit("usage: python oracle/gen_golden.py <reference checkout>/src")
    main(sys.argv[1])
