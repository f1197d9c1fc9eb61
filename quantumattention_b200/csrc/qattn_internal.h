// Internal declarations shared by the translation units of libqattn_sm100.so.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/qattn.h"

#include <atomic>
#include <cstdlib>

namespace qa {

// Per-device one-time state.  Function attributes (dynamic shared-memory opt-in, carve-out) and the SM count belong to
// a device, not to the process: one process may drive several GPUs (SURVEY.md section 8b "threading / streams").
constexpr int kMaxDevices = 64;
inline int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    return dev;
}
// A set of device ordinals ("has X been done on device d"); racing threads set the same bit.
struct DeviceSet {
    std::atomic<unsigned long long> bits{0};
    bool has(int dev) const { return dev >= 0 && dev < kMaxDevices && ((bits.load(std::memory_order_acquire) >> dev) & 1ull); }
    void add(int dev) {
        if (dev >= 0 && dev < kMaxDevices) bits.fetch_or(1ull << dev, std::memory_order_release);
    }
};
// SM count of the current device (cached per ordinal; 0 if the query fails)
inline int sm_count() {
    static std::atomic<int> cache[kMaxDevices];
    const int dev = current_device();
    if (dev >= 0 && dev < kMaxDevices) {
        const int c = cache[dev].load(std::memory_order_relaxed);
        if (c > 0) return c;
    }
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    if (dev >= 0 && dev < kMaxDevices) cache[dev].store(n, std::memory_order_relaxed);
    return n;
}

// Launch with programmatic stream serialisation (programmatic dependent launch): the kernel may be scheduled while the
// previous kernel of the stream is still draining, and synchronises with it through griddepcontrol.wait (ptx.cuh).
// QA_PDL=0 in the environment falls back to ordinary launches (developer switch for A/B runs).
inline bool pdl_enabled() {
    static const bool on = [] {
        const char* e = std::getenv("QA_PDL");
        return !(e && e[0] == '0');
    }();
    return on;
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}


struct QuantArgs {
    const void* x[3];
    void* x8[3];
    float* scale[3];
    int64_t strides[3][4];
    int S[3];
    int B, H, D;
    unsigned int* ctl;  // workspace words 0..7: generation of the last single-pass call, CTA check-in counter
    float* cells;       // workspace + 8: amax cells of the two-pass kernels, then the single-pass kernel's slots
    int rows_per_cta;
    int force_two_pass;
    int given_scale;  // QA_SCALE_HEAD_GIVEN: scale[] is an input
    int amax_only;    // QA_SCALE_HEAD_AMAX_ONLY: write scale[] only
    size_t ws_floats;
    int ws_persistent;  // QA_WS_PERSISTENT: no per-call clear of the single-pass kernel's slots
};

struct AttnArgs {
    const void* q8;
    const void* k8;
    const void* v;
    const float* scale_q;
    const float* scale_k;
    const float* scale_v;
    void* out;
    float* lse;
    int B, Hq, Hkv, Sq, Skv, D;
    int causal;
    float sm_scale;
    int scale_mode;
    int p_mode;
    int v_dtype;
    int out_dtype;
    int qk_dtype;  // QA_DT_E4M3 (FP8 path) or QA_DT_BF16 / QA_DT_FP16 (16-bit path)
    int64_t qs[3], ks[3], vs[3];  // element strides (batch, head, row) of q8 / k8 / v; the last dim is contiguous
    const unsigned* kv_ready = nullptr;  // gated launch: see AttnParams
    int gate_heads = 1, gate_flags = 0;
};

struct MergeArgs {
    float* o_acc;
    float* lse_acc;
    const void* o_new;
    const float* lse_new;
    void* out;
    long long rows;
    int D;
    int dtype;
    int first;
};

int set_error(int code, const char* fmt, ...);
int set_cuda_error(const char* what, cudaError_t e);

int quantize_dispatch(QuantArgs& a, int x_dtype, int scale_mode, int n_tensors, cudaStream_t stream, int* launches);
int attn_fwd_dispatch(const AttnArgs& a, cudaStream_t stream, int* launches);    // e4m3 Q / K
int attn16_fwd_dispatch(const AttnArgs& a, cudaStream_t stream, int* launches);  // bf16 / fp16 Q / K
int merge_dispatch(const MergeArgs& a, cudaStream_t stream, int* launches);

}  // namespace qa
