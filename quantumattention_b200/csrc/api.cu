// extern "C" surface of libqattn_sm100.so (declared in include/qattn.h): argument validation, error reporting,
// and dispatch into the kernels.  No torch types, no allocation, no host synchronisation.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cuda.h>
#include <mutex>
#include "qattn_internal.h"

namespace qa {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
int set_cuda_error(const char* what, cudaError_t e) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return QA_ERR_CUDA;
}

static int check_device() {
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return set_error(QA_ERR_DEVICE, "no CUDA device: %s", cudaGetErrorString(e));
    int major = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) return set_cuda_error("cudaDeviceGetAttribute", e);
    if (major != 10)
        return set_error(QA_ERR_DEVICE, "device %d has compute capability %d.x; this library only runs on sm_100", dev,
                         major);
    return QA_OK;
}

// Element strides (batch, head, row) of a [B, H, S, D] tensor whose last dim is contiguous; NULL = dense.  TMA wants
// every stride a multiple of 16 bytes; dims of size 1 take the dense value (frameworks report arbitrary ones there).
static int take_strides(int64_t (&dst)[3], const int64_t* src, int B, int H, int S, int D, int elem_bytes,
                        const char* name) {
    const int64_t dense[3] = {int64_t(H) * S * D, int64_t(S) * D, int64_t(D)};
    const int sizes[3] = {B, H, S};
    for (int i = 0; i < 3; ++i) {
        dst[i] = (src && sizes[i] > 1) ? src[i] : dense[i];
        if (dst[i] <= 0 || (dst[i] * elem_bytes) % 16 != 0)
            return set_error(QA_ERR_INVALID, "%s: stride %d (%lld elements) must be positive and a multiple of 16 bytes",
                             name, i, (long long)dst[i]);
    }
    if (dst[2] < D) return set_error(QA_ERR_INVALID, "%s: row stride %lld is smaller than the head dimension %d", name, (long long)dst[2], D);
    return QA_OK;
}

}  // namespace qa

using namespace qa;

extern "C" {

int qa_abi_version(void) { return QA_ABI_VERSION; }
const char* qa_last_error(void) { return g_err; }
int qa_last_launch_count(void) { return g_launches; }

int qa_device_supported(int dev) {
    int major = 0;
    cudaError_t e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) {
        set_cuda_error("cudaDeviceGetAttribute", e);
        return 0;
    }
    if (major != 10) {
        set_error(QA_ERR_DEVICE, "device %d has compute capability %d.x; sm_100 required", dev, major);
        return 0;
    }
    return 1;
}

size_t qa_quantize_workspace_floats(int B, int H, int max_S, int D) {
    // 8 header words (generation, check-in counter);  two-pass kernels: amax cells [3BH] (+ spare);  single-pass
    // kernel: one 8-byte slot per 32 KB slab of 3 tensors
    if (B < 1 || H < 1 || max_S < 1 || D < 1) return 0;
    const size_t slab_rows = 32768 / (size_t(D) * 2) ? 32768 / (size_t(D) * 2) : 1;
    const size_t slabs = (size_t(max_S) + slab_rows - 1) / slab_rows * 3 * size_t(B) * size_t(H);
    return size_t(8) + size_t(6) * size_t(B) * size_t(H) + 8 + 2 * slabs;
}

static int quantize_call(int n_tensors, const void* const* x, int x_dtype, const int64_t* x_strides, void* const* x8,
                         float* const* scale, float* amax_ws, int B, int H, const int* S, int D, int scale_mode,
                         void* stream) {
    if (n_tensors < 1 || n_tensors > 3) return set_error(QA_ERR_INVALID, "n_tensors must be 1..3, got %d", n_tensors);
    if (!x || !x_strides || !x8 || !scale || !S) return set_error(QA_ERR_INVALID, "null argument array");
    if (x_dtype != QA_DT_BF16 && x_dtype != QA_DT_FP16)
        return set_error(QA_ERR_INVALID, "x_dtype must be bf16 or fp16");
    const bool ws_persistent = (scale_mode & QA_WS_PERSISTENT) != 0;
    scale_mode &= ~QA_WS_PERSISTENT;
    const bool two_pass = scale_mode == QA_SCALE_HEAD_TWO_PASS;
    const bool given = scale_mode == QA_SCALE_HEAD_GIVEN, amax_only = scale_mode == QA_SCALE_HEAD_AMAX_ONLY;
    if (two_pass || given || amax_only || scale_mode == QA_SCALE_HEAD_RELOAD) scale_mode = QA_SCALE_HEAD;
    if (scale_mode != QA_SCALE_HEAD && scale_mode != QA_SCALE_TOKEN)
        return set_error(QA_ERR_INVALID, "Unsupported scaling_method code: %d", scale_mode);
    if (D != 64 && D != 128 && D != 256) return set_error(QA_ERR_INVALID, "Unsupported head dimension: %d", D);
    if (B < 1 || H < 1 || int64_t(B) * H > 65535) return set_error(QA_ERR_INVALID, "B*H out of range");
    if (scale_mode == QA_SCALE_HEAD && !given && !amax_ws) return set_error(QA_ERR_INVALID, "amax_ws required for head-wise");
    if (reinterpret_cast<uintptr_t>(amax_ws) & 7) return set_error(QA_ERR_INVALID, "amax_ws must be 8-byte aligned");
    QuantArgs a;
    memset(&a, 0, sizeof(a));
    for (int i = 0; i < n_tensors; ++i) {
        if (!x[i] || (!x8[i] && !amax_only) || !scale[i])
            return set_error(QA_ERR_INVALID, "null tensor pointer (tensor %d)", i);
        if (S[i] < 1) return set_error(QA_ERR_INVALID, "empty sequence (tensor %d)", i);
        const int64_t* st = x_strides + 4 * i;
        if (st[3] != 1) return set_error(QA_ERR_INVALID, "last-dim stride must be 1 (tensor %d)", i);
        if ((reinterpret_cast<uintptr_t>(x[i]) & 15) || (st[0] & 7) || (st[1] & 7) || (st[2] & 7))
            return set_error(QA_ERR_INVALID, "rows must be 16-byte aligned (tensor %d)", i);
        if (!amax_only && (reinterpret_cast<uintptr_t>(x8[i]) & 15)) return set_error(QA_ERR_INVALID, "x8 must be 16-byte aligned");
        a.x[i] = x[i];
        a.x8[i] = x8[i];
        a.scale[i] = scale[i];
        for (int d = 0; d < 4; ++d) a.strides[i][d] = st[d];
        a.S[i] = S[i];
    }
    a.B = B, a.H = H, a.D = D;
    a.ctl = reinterpret_cast<unsigned int*>(amax_ws);
    a.cells = amax_ws ? amax_ws + 8 : nullptr;
    a.force_two_pass = two_pass ? 1 : 0;
    a.given_scale = given ? 1 : 0;
    a.amax_only = amax_only ? 1 : 0;
    a.ws_persistent = ws_persistent ? 1 : 0;
    int max_S = 0;
    for (int i = 0; i < n_tensors; ++i) max_S = S[i] > max_S ? S[i] : max_S;
    a.ws_floats = qa_quantize_workspace_floats(B, H, max_S, D);
    int rc = check_device();
    if (rc != QA_OK) return rc;
    return quantize_dispatch(a, x_dtype, scale_mode, n_tensors, static_cast<cudaStream_t>(stream), &g_launches);
}

int qa_quantize_fp8(int n_tensors, const void* const* x, int x_dtype, const int64_t* x_strides, void* const* x8,
                    float* const* scale, float* amax_ws, int B, int H, const int* S, int D, int scale_mode,
                    void* stream) {
    g_launches = 0;
    return quantize_call(n_tensors, x, x_dtype, x_strides, x8, scale, amax_ws, B, H, S, D, scale_mode, stream);
}

static int fp8_attn_call(const void* q8, const void* k8, const void* v, int v_dtype, const int64_t* q_strides,
                         const int64_t* k_strides, const int64_t* v_strides, const float* scale_q, const float* scale_k,
                         const float* scale_v, int scale_mode, void* out, int out_dtype, float* lse, int B, int Hq,
                         int Hkv, int Sq, int Skv, int D, int causal, float sm_scale, int p_mode, void* stream,
                         const unsigned* kv_ready = nullptr, int gate_heads = 1, int gate_flags = 0) {
    if (!q8 || !k8 || !v || !scale_q || !scale_k || !out) return set_error(QA_ERR_INVALID, "null pointer argument");
    if (kv_ready && (gate_heads < 1 || gate_flags < 1 || gate_flags > 64))
        return set_error(QA_ERR_INVALID, "gated launch: heads_per_gate >= 1 and 1 <= flags_per_gate <= 64 expected");
    if (D != 64 && D != 128 && D != 256) return set_error(QA_ERR_INVALID, "Unsupported head dimension: %d", D);
    if (B < 1 || Hq < 1 || Hkv < 1 || Sq < 1 || Skv < 1) return set_error(QA_ERR_INVALID, "empty problem");
    if (Hq % Hkv != 0)
        return set_error(QA_ERR_INVALID, "Expect Hq to be a multiple of Hkv but got Hq=%d and Hkv=%d.", Hq, Hkv);
    if (Hq > 65535 || B > 65535) return set_error(QA_ERR_INVALID, "B or Hq exceeds the grid limit 65535");
    if (scale_mode != QA_SCALE_HEAD && scale_mode != QA_SCALE_TOKEN)
        return set_error(QA_ERR_INVALID, "Unsupported scaling_method code: %d", scale_mode);
    if (out_dtype != QA_DT_BF16 && out_dtype != QA_DT_FP16)
        return set_error(QA_ERR_INVALID, "out_dtype must be bf16 or fp16");
    if (!(sm_scale > 0.f) || !(sm_scale < 1e30f)) return set_error(QA_ERR_INVALID, "sm_scale must be positive");
    if (p_mode == QA_P_16BIT) {
        if (v_dtype != QA_DT_BF16 && v_dtype != QA_DT_FP16)
            return set_error(QA_ERR_INVALID, "p_mode 16BIT needs a bf16/fp16 value tensor");
        if (v_dtype != out_dtype) return set_error(QA_ERR_INVALID, "p_mode 16BIT: out_dtype must equal v_dtype");
    } else if (p_mode == QA_P_E4M3 || p_mode == QA_P_E4M3_HILO) {
        if (v_dtype != QA_DT_E4M3) return set_error(QA_ERR_INVALID, "FP8 P modes need an e4m3 value tensor");
        if (!scale_v) return set_error(QA_ERR_INVALID, "scale_v required for an e4m3 value tensor");
    } else {
        return set_error(QA_ERR_INVALID, "unknown p_mode %d", p_mode);
    }
    if ((reinterpret_cast<uintptr_t>(q8) | reinterpret_cast<uintptr_t>(k8) | reinterpret_cast<uintptr_t>(v)) & 15)
        return set_error(QA_ERR_INVALID, "tensor base pointers must be 16-byte aligned");
    if (reinterpret_cast<uintptr_t>(out) & 31) return set_error(QA_ERR_INVALID, "out must be 32-byte aligned");
    AttnArgs a;
    int rc;
    if ((rc = take_strides(a.qs, q_strides, B, Hq, Sq, D, 1, "q8")) != QA_OK) return rc;
    if ((rc = take_strides(a.ks, k_strides, B, Hkv, Skv, D, 1, "k8")) != QA_OK) return rc;
    if ((rc = take_strides(a.vs, v_strides, B, Hkv, Skv, D, p_mode == QA_P_16BIT ? 2 : 1, "v")) != QA_OK) return rc;
    if ((rc = check_device()) != QA_OK) return rc;
    a.q8 = q8, a.k8 = k8, a.v = v;
    a.scale_q = scale_q, a.scale_k = scale_k, a.scale_v = scale_v;
    a.out = out, a.lse = lse;
    a.B = B, a.Hq = Hq, a.Hkv = Hkv, a.Sq = Sq, a.Skv = Skv, a.D = D;
    a.causal = causal ? 1 : 0;
    a.sm_scale = sm_scale;
    a.scale_mode = scale_mode;
    a.p_mode = p_mode;
    a.v_dtype = v_dtype;
    a.out_dtype = out_dtype;
    a.qk_dtype = QA_DT_E4M3;
    a.kv_ready = kv_ready, a.gate_heads = gate_heads, a.gate_flags = kv_ready ? gate_flags : 0;
    return attn_fwd_dispatch(a, static_cast<cudaStream_t>(stream), &g_launches);
}

int qa_fp8_attn_fwd_gated(const void* q8, const void* k8, const void* v, int v_dtype, const int64_t* q_strides,
                          const int64_t* k_strides, const int64_t* v_strides, const float* scale_q, const float* scale_k,
                          const float* scale_v, int scale_mode, void* out, int out_dtype, float* lse, int B, int Hq,
                          int Hkv, int Sq, int Skv, int D, int causal, float sm_scale, int p_mode,
                          const unsigned* kv_ready, int heads_per_gate, int flags_per_gate, void* stream) {
    g_launches = 0;
    if (!kv_ready) return set_error(QA_ERR_INVALID, "null pointer argument");
    return fp8_attn_call(q8, k8, v, v_dtype, q_strides, k_strides, v_strides, scale_q, scale_k, scale_v, scale_mode, out,
                         out_dtype, lse, B, Hq, Hkv, Sq, Skv, D, causal, sm_scale, p_mode, stream, kv_ready,
                         heads_per_gate, flags_per_gate);
}

int qa_set_flag(unsigned* flag, void* stream) {
    g_launches = 0;
    if (!flag) return set_error(QA_ERR_INVALID, "null pointer argument");
    // A stream memory operation (cuStreamWriteValue32): performed by the stream's front end in stream order behind the
    // copies it vouches for.  NOT cudaMemsetAsync: a small memset is a kernel, and the gated attention kernel it would
    // release holds every SM (one CTA per SM, the whole register file) while it polls - the memset would never run.
    typedef CUresult (*PFN_write32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
    static PFN_write32 fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_write32>(p);
    });
    if (!fn) return set_error(QA_ERR_DEVICE, "cuStreamWriteValue32 is unavailable (no CUDA driver?)");
    int rc = check_device();
    if (rc != QA_OK) return rc;
    CUresult r = fn(static_cast<CUstream>(stream), reinterpret_cast<CUdeviceptr>(flag), 0x01010101u, 0u);
    if (r != CUDA_SUCCESS) return set_error(QA_ERR_CUDA, "cuStreamWriteValue32 failed with CUresult %d", int(r));
    return QA_OK;
}

int qa_fp8_attn_fwd(const void* q8, const void* k8, const void* v, int v_dtype, const int64_t* q_strides,
                    const int64_t* k_strides, const int64_t* v_strides, const float* scale_q, const float* scale_k,
                    const float* scale_v, int scale_mode, void* out, int out_dtype, float* lse, int B, int Hq, int Hkv,
                    int Sq, int Skv, int D, int causal, float sm_scale, int p_mode, void* stream) {
    g_launches = 0;
    return fp8_attn_call(q8, k8, v, v_dtype, q_strides, k_strides, v_strides, scale_q, scale_k, scale_v, scale_mode, out,
                         out_dtype, lse, B, Hq, Hkv, Sq, Skv, D, causal, sm_scale, p_mode, stream);
}

int qa_fp8_attn_func(const void* q, const void* k, const void* v, int dtype, const int64_t* q_strides,
                     const int64_t* k_strides, const int64_t* v_strides, void* q8, void* k8, void* v8, float* scale_q,
                     float* scale_k, float* scale_v, float* amax_ws, int ws_flags, void* out, float* lse, int B, int Hq,
                     int Hkv, int Sq, int Skv, int D, int causal, float sm_scale, int scale_mode, int p_mode,
                     void* stream) {
    g_launches = 0;
    if (!q || !k || !v || !q8 || !k8 || !scale_q || !scale_k || !out) return set_error(QA_ERR_INVALID, "null pointer argument");
    if (scale_mode != QA_SCALE_HEAD && scale_mode != QA_SCALE_TOKEN)
        return set_error(QA_ERR_INVALID, "Unsupported scaling_method code: %d", scale_mode);
    if (ws_flags & ~QA_WS_PERSISTENT) return set_error(QA_ERR_INVALID, "ws_flags may only carry QA_WS_PERSISTENT");
    const bool v_fp8 = p_mode != QA_P_16BIT;
    if (v_fp8 && (!v8 || !scale_v)) return set_error(QA_ERR_INVALID, "FP8 P modes need v8 and scale_v buffers");
    if (B < 1 || Hq < 1 || Hkv < 1) return set_error(QA_ERR_INVALID, "empty problem");
    // strides as the quantiser wants them: 4 per tensor, the last one 1
    auto four = [](int64_t (&d)[4], const int64_t* s, int H, int S, int D) {
        d[0] = s ? s[0] : int64_t(H) * S * D, d[1] = s ? s[1] : int64_t(S) * D, d[2] = s ? s[2] : int64_t(D), d[3] = 1;
    };
    int64_t st[3][4];
    four(st[0], q_strides, Hq, Sq, D);
    four(st[1], k_strides, Hkv, Skv, D);
    four(st[2], v_strides, Hkv, Skv, D);
    int rc;
    // one quantiser launch for everything that shares a head count (head-wise V rides along with K; token-wise Q / K
    // scales leave V, whose scale is always per head, to a launch of its own)
    const bool v_with_k = v_fp8 && scale_mode == QA_SCALE_HEAD;
    if (Hq == Hkv) {
        const void* x[3] = {q, k, v};
        void* x8[3] = {q8, k8, v8};
        float* sc[3] = {scale_q, scale_k, scale_v};
        const int S[3] = {Sq, Skv, Skv};
        rc = quantize_call(v_with_k ? 3 : 2, x, dtype, &st[0][0], x8, sc, amax_ws, B, Hq, S, D, scale_mode | ws_flags, stream);
        if (rc != QA_OK) return rc;
    } else {
        const void* xq[1] = {q};
        void* xq8[1] = {q8};
        float* sq[1] = {scale_q};
        const int Sq1[1] = {Sq};
        rc = quantize_call(1, xq, dtype, &st[0][0], xq8, sq, amax_ws, B, Hq, Sq1, D, scale_mode | ws_flags, stream);
        if (rc != QA_OK) return rc;
        const void* x[2] = {k, v};
        void* x8[2] = {k8, v8};
        float* sc[2] = {scale_k, scale_v};
        const int S[2] = {Skv, Skv};
        rc = quantize_call(v_with_k ? 2 : 1, x, dtype, &st[1][0], x8, sc, amax_ws, B, Hkv, S, D, scale_mode | ws_flags, stream);
        if (rc != QA_OK) return rc;
    }
    if (v_fp8 && !v_with_k) {
        const void* x[1] = {v};
        void* x8[1] = {v8};
        float* sc[1] = {scale_v};
        const int S[1] = {Skv};
        rc = quantize_call(1, x, dtype, &st[2][0], x8, sc, amax_ws, B, Hkv, S, D, QA_SCALE_HEAD | ws_flags, stream);
        if (rc != QA_OK) return rc;
    }
    return fp8_attn_call(q8, k8, v_fp8 ? v8 : v, v_fp8 ? QA_DT_E4M3 : dtype, nullptr, nullptr, v_fp8 ? nullptr : v_strides,
                         scale_q, scale_k, v_fp8 ? scale_v : nullptr, scale_mode, out, dtype, lse, B, Hq, Hkv, Sq, Skv, D,
                         causal, sm_scale, p_mode, stream);
}

int qa_attn_fwd(const void* q, const void* k, const void* v, int dtype, const int64_t* q_strides,
                const int64_t* k_strides, const int64_t* v_strides, void* out, float* lse, int B, int Hq, int Hkv, int Sq,
                int Skv, int D, int causal, float sm_scale, void* stream) {
    g_launches = 0;
    if (!q || !k || !v || !out) return set_error(QA_ERR_INVALID, "null pointer argument");
    if (dtype != QA_DT_BF16 && dtype != QA_DT_FP16)
        return set_error(QA_ERR_INVALID, "Expected query, key, and value to have dtype fp16 or bf16 (code %d)", dtype);
    if (D != 64 && D != 128 && D != 256) return set_error(QA_ERR_INVALID, "Unsupported head dimension: %d", D);
    if (B < 1 || Hq < 1 || Hkv < 1 || Sq < 1 || Skv < 1) return set_error(QA_ERR_INVALID, "empty problem");
    if (Hq % Hkv != 0)
        return set_error(QA_ERR_INVALID, "Expect Hq to be a multiple of Hkv but got Hq=%d and Hkv=%d.", Hq, Hkv);
    if (Hq > 65535 || B > 65535) return set_error(QA_ERR_INVALID, "B or Hq exceeds the grid limit 65535");
    if (!(sm_scale > 0.f) || !(sm_scale < 1e30f)) return set_error(QA_ERR_INVALID, "sm_scale must be positive");
    if ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) & 15)
        return set_error(QA_ERR_INVALID, "tensor base pointers must be 16-byte aligned");
    if (reinterpret_cast<uintptr_t>(out) & 31) return set_error(QA_ERR_INVALID, "out must be 32-byte aligned");
    AttnArgs a;
    int rc;
    if ((rc = take_strides(a.qs, q_strides, B, Hq, Sq, D, 2, "q")) != QA_OK) return rc;
    if ((rc = take_strides(a.ks, k_strides, B, Hkv, Skv, D, 2, "k")) != QA_OK) return rc;
    if ((rc = take_strides(a.vs, v_strides, B, Hkv, Skv, D, 2, "v")) != QA_OK) return rc;
    if ((rc = check_device()) != QA_OK) return rc;
    a.q8 = q, a.k8 = k, a.v = v;
    a.scale_q = a.scale_k = a.scale_v = nullptr;
    a.out = out, a.lse = lse;
    a.B = B, a.Hq = Hq, a.Hkv = Hkv, a.Sq = Sq, a.Skv = Skv, a.D = D;
    a.causal = causal ? 1 : 0;
    a.sm_scale = sm_scale;
    a.scale_mode = QA_SCALE_HEAD;
    a.p_mode = QA_P_16BIT;
    a.v_dtype = a.out_dtype = a.qk_dtype = dtype;
    return attn16_fwd_dispatch(a, static_cast<cudaStream_t>(stream), &g_launches);
}

int qa_copy_2d(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width_bytes, size_t rows,
               void* stream) {
    g_launches = 0;
    if (!dst || !src) return set_error(QA_ERR_INVALID, "null pointer argument");
    if (width_bytes == 0 || rows == 0) return QA_OK;
    if (dst_pitch < width_bytes || src_pitch < width_bytes) return set_error(QA_ERR_INVALID, "pitch smaller than the row width");
    // cudaMemcpyDefault: source and destination are told apart by their addresses (unified addressing), so a
    // peer-mapped source makes this a copy-engine transfer over NVLink that occupies no SM
    cudaError_t e = cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, width_bytes, rows, cudaMemcpyDefault,
                                      static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return set_cuda_error("cudaMemcpy2DAsync", e);
    return QA_OK;
}

int qa_copy_2d_batch(int n, void* const* dst, const size_t* dst_pitch, const void* const* src, const size_t* src_pitch,
                     const size_t* width_bytes, const size_t* rows, void* const* streams) {
    g_launches = 0;
    if (n < 0 || (n > 0 && (!dst || !dst_pitch || !src || !src_pitch || !width_bytes || !rows || !streams)))
        return set_error(QA_ERR_INVALID, "null argument array");
    for (int i = 0; i < n; ++i) {
        int rc = qa_copy_2d(dst[i], dst_pitch[i], src[i], src_pitch[i], width_bytes[i], rows[i], streams[i]);
        if (rc != QA_OK) return rc;
    }
    return QA_OK;
}

int qa_merge_partials(float* o_acc, float* lse_acc, const void* o_new, int o_dtype, const float* lse_new, void* out,
                      long long rows, int D, int first, void* stream) {
    g_launches = 0;
    if (!lse_acc || !o_new || !lse_new) return set_error(QA_ERR_INVALID, "null pointer argument");
    if (!o_acc && !(first && out)) return set_error(QA_ERR_INVALID, "o_acc may only be NULL when first != 0 and out is given");
    if (o_dtype != QA_DT_BF16 && o_dtype != QA_DT_FP16) return set_error(QA_ERR_INVALID, "o_dtype must be bf16 or fp16");
    if (D != 64 && D != 128 && D != 256) return set_error(QA_ERR_INVALID, "Unsupported head dimension: %d", D);
    if (rows < 1) return set_error(QA_ERR_INVALID, "empty problem");
    if ((reinterpret_cast<uintptr_t>(o_acc) | reinterpret_cast<uintptr_t>(o_new) | reinterpret_cast<uintptr_t>(out)) & 15)
        return set_error(QA_ERR_INVALID, "tensor base pointers must be 16-byte aligned");
    int rc = check_device();
    if (rc != QA_OK) return rc;
    MergeArgs a;
    a.o_acc = o_acc, a.lse_acc = lse_acc, a.o_new = o_new, a.lse_new = lse_new, a.out = out;
    a.rows = rows, a.D = D, a.dtype = o_dtype, a.first = first ? 1 : 0;
    return merge_dispatch(a, static_cast<cudaStream_t>(stream), &g_launches);
}

}  // extern "C"
