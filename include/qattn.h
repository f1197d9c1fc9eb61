/* qattn.h - C ABI of the B200-native FP8 fused-attention library (libqattn_sm100.so).
 *
 * This is the drop-in boundary for the hot path of WaveSpeedAI/QuantumAttention: everything below the Python
 * functions `fp8_attn_func` / `fp8_token_wise_attn_func` / `dynamically_quantize_fp8`.  The reference has no C
 * ABI; its boundary is a JIT-built torch extension exposing
 *     attention_forward(q, k, v[, scale_q, scale_k], causal) -> [o]
 * (reference: src/quantum_attn/tk/attention.py:355-360, launcher :362-647) plus Inductor-generated quantise kernels
 * (reference: src/quantum_attn/nn.py:14-19, 410-418).  Each entry point below cites what it replaces.
 *
 * Conventions
 *   - plain pointers to DEVICE memory, sizes as int, no torch types; the caller owns every buffer
 *   - every call is asynchronous on the given stream; no host sync, no allocation inside the library
 *   - return value: 0 = ok, negative = error (see QA_ERR_*); text via qa_last_error() (thread-local)
 *   - tensors are [B, H, S, D] with D contiguous; inputs may carry batch / head / row strides (a [B,S,H,D]-held
 *     tensor is consumed in place through TMA); tensors the library WRITES are dense ([B,H,S,D] contiguous)
 *   - the library requires an sm_100 device; there is no fallback path
 */
#ifndef QATTN_H_
#define QATTN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QA_ABI_VERSION 6

/* element types */
#define QA_DT_BF16 0
#define QA_DT_FP16 1
#define QA_DT_E4M3 2

/* scale granularity (reference: "head-wise" src/quantum_attn/nn.py:411-412, "token-wise" :413-414) */
#define QA_SCALE_HEAD 0  /* one fp32 scale per (b, h):        scale[B*H]     */
#define QA_SCALE_TOKEN 1 /* one fp32 scale per (b, h, token): scale[B*H*S]   */
#define QA_SCALE_HEAD_TWO_PASS 2 /* qa_quantize_fp8 only: QA_SCALE_HEAD results through the two-pass kernels (the path
                                    heads longer than one resident wave take by themselves); for tests */

#define QA_SCALE_HEAD_AMAX_ONLY 3 /* qa_quantize_fp8 only: write scale[] (from the local amax), touch no x8 (may be NULL) */
#define QA_SCALE_HEAD_GIVEN 4     /* qa_quantize_fp8 only: scale[] is an INPUT; quantise with it.  The pair lets a caller
                                    that shards one sequence over several GPUs take the MAX of the per-shard scales
                                    (scale is monotone in amax) and obtain the bytes the unsharded call would produce */

#define QA_SCALE_HEAD_RELOAD 5    /* accepted for ABI 6 compatibility; same as QA_SCALE_HEAD */

#define QA_WS_PERSISTENT 0x100    /* qa_quantize_fp8, OR-ed into scale_mode: amax_ws was zero-filled ONCE by the caller
                                    when it was allocated and has since been written only by this library (calls of any
                                    shape it is large enough for, all ordered on one stream).  The single-pass head-wise
                                    kernel then skips its per-call clear: its rendezvous slots carry a per-call
                                    generation tag, and older tags never match.  The generation is kept in the workspace
                                    itself (word 0) and advanced by the kernel, so a call captured into a CUDA graph
                                    takes a fresh tag on every replay.  Without the flag the workspace is plain scratch
                                    whose contents are ignored (it is cleared by every call). */

/* how P = softmax(QK^T) is fed to the second GEMM */
#define QA_P_E4M3 0      /* P -> e4m3, V e4m3, tcgen05 kind::f8f6f4               (north-star fast path)          */
#define QA_P_E4M3_HILO 1 /* P -> e4m3 hi + e4m3 lo (two MMAs), V e4m3            (accurate FP8 path)             */
#define QA_P_16BIT 2     /* P -> bf16/fp16, V unquantised 16-bit, kind::f16       (the reference's own numerics:  */
                         /*                                   src/quantum_attn/tk/attention.py:230,286,318)      */

/* error codes */
#define QA_OK 0
#define QA_ERR_INVALID (-1)     /* bad argument / unsupported shape */
#define QA_ERR_DEVICE (-2)      /* device is not sm_100, or driver entry point missing */
#define QA_ERR_CUDA (-3)        /* CUDA runtime error at launch */
#define QA_ERR_UNSUPPORTED (-4) /* valid request this build does not implement yet */

int qa_abi_version(void);
const char* qa_last_error(void);

/* 1 if device `dev` can run the kernels (compute capability 10.x), else 0 (and qa_last_error says why).
 * Replaces the reference's capability gate (src/quantum_attn/nn.py:208-216), which accepts >= 9.0 although its
 * kernel only exists for sm_90a. */
int qa_device_supported(int dev);

/* Dynamic FP8 quantisation, one launch pair for up to 3 tensors of the same [B,H,*,D] family.
 *   scale = max(amax(|x|) * (1/448), FLT_EPSILON);  x8 = e4m3_rne(clamp(x / scale, +-448))   (all fp32, IEEE division)
 * Replaces the Inductor-generated kernels of `_dynamically_quantize_fp8` (reference: src/quantum_attn/nn.py:14-19).
 *
 *   n_tensors   1..3
 *   x[i]        device pointer, dtype x_dtype (QA_DT_BF16 / QA_DT_FP16), logical shape [B, H, S[i], D]
 *   x_strides   4 element strides per tensor (x_strides[4*i .. 4*i+3]); the last one must be 1, rows 16-byte aligned
 *   x8[i]       out: dense e4m3 bytes [B, H, S[i], D]
 *   scale[i]    out: fp32 [B*H] (QA_SCALE_HEAD) or [B*H*S[i]] (QA_SCALE_TOKEN)
 *   amax_ws     scratch of qa_quantize_workspace_floats(B, H, max_i S[i], D) floats, 8-byte aligned (head-wise only;
 *               may be NULL for token mode); need not be zeroed (but see QA_WS_PERSISTENT), must not be shared by
 *               calls that can run concurrently.  The single-pass head-wise kernel (one CTA per SM, CTAs rendezvous
 *               through this workspace) needs its whole grid resident at once: it is launched with the cooperative
 *               attribute, so it is only scheduled once the grid fits (concurrent calls on other streams queue), and
 *               a bounded poll turns any remaining non-resident grid into a trap rather than a hang.
 */
size_t qa_quantize_workspace_floats(int B, int H, int max_S, int D);
int qa_quantize_fp8(int n_tensors, const void* const* x, int x_dtype, const int64_t* x_strides, void* const* x8,
                    float* const* scale, float* amax_ws, int B, int H, const int* S, int D, int scale_mode,
                    void* stream);

/* Fused QK^T -> online softmax -> PV forward on quantised inputs.
 * Replaces `attention_forward` of the reference's TK module (src/quantum_attn/tk/attention.py:355-647) and the kernel
 * it launches (`fwd_attend_ker`, :97-349), and defines the same function as the op
 * `quantum_attn::fp8_attention_forward` (src/quantum_attn/ops.py:64-95):
 *     out = softmax(sm_scale * (q8*scale_q)(k8*scale_k)^T  [+ top-left causal mask]) (v*scale_v)
 *
 *   q8, k8      e4m3 [B,Hq,Sq,D], [B,Hkv,Skv,D]
 *   v           QA_P_E4M3 / QA_P_E4M3_HILO: e4m3 [B,Hkv,Skv,D] with scale_v[B*Hkv] (head-wise)
 *               QA_P_16BIT: bf16/fp16 (v_dtype) [B,Hkv,Skv,D], scale_v may be NULL
 *   q_strides, k_strides, v_strides
 *               3 ELEMENT strides each - (batch, head, row) - or NULL for a dense tensor; D is contiguous; every stride
 *               a multiple of 16 bytes.  The tensor maps are built from them, so a [B,S,H,D]-held tensor is read in
 *               place (the reference copies it dense first, src/quantum_attn/tk/attention.py:419-421)
 *   scale_q/k   fp32, layout per scale_mode (token mode: scale_q[B*Hq*Sq], scale_k[B*Hkv*Skv])
 *   out         dense [B,Hq,Sq,D] of out_dtype (QA_DT_BF16 / QA_DT_FP16), 32-byte aligned
 *   lse         optional fp32 [B*Hq*Sq]: natural-log sum-exp of the scaled scores per row (for merging partial
 *               results across sequence shards); NULL to skip.  The reference leaves this output commented out
 *               (src/quantum_attn/tk/attention.py:333-346).  In QA_P_E4M3 mode the sum is taken over the probabilities
 *               as rounded to e4m3 - the weights that multiply V and normalise `out` - so it can differ from the
 *               exact log-sum-exp by up to ln(1 + 2^-4) ~= 0.061, plus ~2e-3 from the exponentials.  That bound holds
 *               while the keys whose weight falls under e4m3's normal range (more than 10 log2 units below the row
 *               maximum) carry a negligible share of the row sum; it is reached by a row dominated by one key whose
 *               weight sits up to TAU = 4 log2 units above the stale running maximum.  Merging partial results with
 *               it reproduces the one-launch result.
 *   sm_scale    softmax scale; pass 1/sqrt(D) for the reference's behaviour (src/quantum_attn/tk/attention.py:208-210)
 *   Hq % Hkv == 0 (GQA: kv head = q head / (Hq/Hkv)); D in {64, 128, 256}; causal mask is top-left aligned.
 */
int qa_fp8_attn_fwd(const void* q8, const void* k8, const void* v, int v_dtype, const int64_t* q_strides,
                    const int64_t* k_strides, const int64_t* v_strides, const float* scale_q, const float* scale_k,
                    const float* scale_v, int scale_mode, void* out, int out_dtype, float* lse, int B, int Hq, int Hkv,
                    int Sq, int Skv, int D, int causal, float sm_scale, int p_mode, void* stream);

/* qa_fp8_attn_fwd as a GATED launch: the kernel starts at once, but the CTAs of kv head h read K / V only after the
 * `flags_per_gate` 32-bit words kv_ready[(h / heads_per_gate) * flags_per_gate ...] are all non-zero.  The caller
 * zero-fills the words on the launch stream before the call and sets each one with qa_set_flag on whatever stream
 * brings that group of heads (one word per stream that carries a part of it).  New operator (the reference never
 * shards a sequence): the sequence-sharded path attends ALL heads in ONE launch while the other ranks' K / V blocks
 * of the later heads are still crossing NVLink on the copy engines - one launch keeps the hardware's dynamic CTA
 * dispatch (fast SMs take more CTAs), where one launch per head group ran the groups in lock-step waves (each group
 * waiting for the slowest CTA of the one before it: +12 % at 148 CTAs per group, profiles/r02_wave_probe.txt).
 * Q must be complete in stream order (it is local).  Only for transfers that need no SM (copy engines): a transfer
 * KERNEL could find every SM held by a polling CTA.  A flag that never arrives traps the kernel after ~4 s of polling.
 */
int qa_fp8_attn_fwd_gated(const void* q8, const void* k8, const void* v, int v_dtype, const int64_t* q_strides,
                          const int64_t* k_strides, const int64_t* v_strides, const float* scale_q, const float* scale_k,
                          const float* scale_v, int scale_mode, void* out, int out_dtype, float* lse, int B, int Hq,
                          int Hkv, int Sq, int Skv, int D, int causal, float sm_scale, int p_mode,
                          const unsigned* kv_ready, int heads_per_gate, int flags_per_gate, void* stream);
/* *flag = non-zero in stream order, as a stream memory operation (cuStreamWriteValue32): no kernel, no SM - a kernel
 * could never run while the gated launch it is to release holds every SM. */
int qa_set_flag(unsigned* flag, void* stream);

/* The whole of `fp8_attn_func` on 16-bit inputs in ONE call: quantise Q and K (and V in the FP8 P modes), then the
 * fused forward.  Replaces `_fp8_attention_wrapper` + the op call of the reference (src/quantum_attn/nn.py:394-430:
 * two `_dynamically_quantize_fp8` + `quantum_attn::fp8_attention_forward`) and saves the host a second crossing of
 * the boundary per attention call.  Same results as qa_quantize_fp8 followed by qa_fp8_attn_fwd.
 *
 *   q, k, v     bf16/fp16 (`dtype`) [B,Hq,Sq,D], [B,Hkv,Skv,D], [B,Hkv,Skv,D] with optional strides as above
 *   q8, k8, v8  scratch for the dense e4m3 tensors (v8 only in the FP8 P modes, else NULL); they hold the quantised
 *               tensors on return, so a caller may keep k8 / v8 and their scales for later qa_fp8_attn_fwd calls
 *   scale_q/k/v out: fp32 scales ([B*H] head-wise, [B*H*S] token-wise for q / k; scale_v always [B*Hkv])
 *   amax_ws     as for qa_quantize_fp8 (sized for max(Hq, Hkv) heads and max(Sq, Skv) rows); ws_flags 0 or QA_WS_PERSISTENT
 *   out         dense [B,Hq,Sq,D] of `dtype`; lse optional
 */
int qa_fp8_attn_func(const void* q, const void* k, const void* v, int dtype, const int64_t* q_strides,
                     const int64_t* k_strides, const int64_t* v_strides, void* q8, void* k8, void* v8, float* scale_q,
                     float* scale_k, float* scale_v, float* amax_ws, int ws_flags, void* out, float* lse, int B, int Hq,
                     int Hkv, int Sq, int Skv, int D, int causal, float sm_scale, int scale_mode, int p_mode,
                     void* stream);

/* The same fused forward with Q and K left in 16 bits: S = Q K^T as tcgen05 kind::f16, P and V 16-bit, fp32
 * accumulation and softmax.  Replaces the reference's non-FP8 TK module - `attention_forward(q, k, v, causal)`
 * (src/quantum_attn/tk/attention.py:355-360 with is_fp8 = false, kernel :238-240,289-313) - behind `attn_func`
 * (src/quantum_attn/quantum_attn_interface.py:41-59) / op `quantum_attn::attention_forward`
 * (src/quantum_attn/ops.py:32-45):
 *     out = softmax(sm_scale * q k^T  [+ top-left causal mask]) v
 *
 *   q, k, v     [B,Hq,Sq,D], [B,Hkv,Skv,D], [B,Hkv,Skv,D], all of `dtype` (QA_DT_BF16 / QA_DT_FP16), optional element
 *               strides (batch, head, row) as in qa_fp8_attn_fwd
 *   out         dense [B,Hq,Sq,D] of `dtype`;  lse as in qa_fp8_attn_fwd (NULL to skip)
 *   Hq % Hkv == 0; D in {64, 128, 256}; causal mask is top-left aligned.
 */
int qa_attn_fwd(const void* q, const void* k, const void* v, int dtype, const int64_t* q_strides,
                const int64_t* k_strides, const int64_t* v_strides, void* out, float* lse, int B, int Hq, int Hkv, int Sq,
                int Skv, int D, int causal, float sm_scale, void* stream);

/* Combine two partial attention results over disjoint key sets, row by row:
 *     m = max(lse_acc, lse_new); w_x = exp(lse_x - m); O = (w_acc O_acc + w_new O_new) / (w_acc + w_new);
 *     LSE = m + log(w_acc + w_new)
 * New operator (the reference never shards a sequence; its kernel leaves the LSE output commented out,
 * src/quantum_attn/tk/attention.py:333-346).  Used by the sequence ring for the long-video shape.
 *
 *   o_acc, lse_acc  running result: fp32 [rows, D] and fp32 [rows]; in/out
 *   o_new, lse_new  partial result of one qa_fp8_attn_fwd call: 16-bit [rows, D] (o_dtype) and fp32 [rows]
 *   out             NULL, or 16-bit [rows, D]: the merged rows are written THERE instead of into o_acc (last step)
 *   first           != 0: the accumulator is uninitialised; the call copies (o_new, lse_new) into it
 *   rows            B * Hq * Sq
 */
int qa_merge_partials(float* o_acc, float* lse_acc, const void* o_new, int o_dtype, const float* lse_new, void* out,
                      long long rows, int D, int first, void* stream);

/* Strided block copy on the copy engines: `rows` rows of `width_bytes`, row r from src + r * src_pitch to
 * dst + r * dst_pitch (cudaMemcpy2DAsync, direction inferred from the addresses).  The sequence-sharded path pulls the
 * other ranks' e4m3 K / V blocks with it straight from PEER memory (buffers mapped through CUDA IPC / symmetric
 * memory) into the per-head layout the fused kernel reads: the transfer crosses NVLink without occupying an SM, so
 * it overlaps the attention kernel completely - a collective kernel would take SMs away from it.  New operator (the
 * reference never shards a sequence).  Asynchronous on `stream`; launches no kernel. */
int qa_copy_2d(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width_bytes, size_t rows,
               void* stream);
/* n such copies in one call (copy i on streams[i]): a head group's blocks from every peer cost the host one crossing
 * of the boundary instead of 2 x world. */
int qa_copy_2d_batch(int n, void* const* dst, const size_t* dst_pitch, const void* const* src, const size_t* src_pitch,
                     const size_t* width_bytes, const size_t* rows, void* const* streams);

/* Number of kernels the previous call on this thread launched (for bench.py's gpu_launches accounting). */
int qa_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* QATTN_H_ */
