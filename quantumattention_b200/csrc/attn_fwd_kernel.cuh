// Fused FP8 attention forward for sm_100a:  S = Q K^T (tcgen05 kind::f8f6f4, fp32 in TMEM)  ->  online softmax in
// registers (one thread per query row, base-2 domain, lazy rescale)  ->  P written back into TMEM as e4m3  ->
// O += P V (tcgen05, A operand from TMEM, V straight from its [kv][D] layout as an MN-major B operand).
//
// What it replaces: `fwd_attend_ker` of the reference (src/quantum_attn/tk/attention.py:97-349) and its launcher
// (:355-647).  Same function (dequant scale folded into the exp2 argument as in :204-210,248-250; top-left causal
// mask as in :252-263, or shifted by a run-time diagonal offset for the bottom-right alignment of the C ABI; ragged
// tails via TMA zero fill + -inf columns as in :269-271), different machine:
//
//   CTA = 2 query tiles of 128 rows, 12 warps (3 warpgroups; setmaxnreg moves registers to the softmax warps):
//     warps 0-3  softmax + (rare) O rescale + epilogue of query tile 0   (thread r <-> TMEM lane r <-> query row r)
//     warps 4-7  the same for query tile 1
//     warp  8/10 MMA issuer of query tile 0 / 1 (one elected thread each)
//     warp  9    TMA producer: Q once, K/V tiles of 128 keys through mbarrier rings      (warp 11 idle)
//   The softmax / MMA hand-off runs in STEPS of 64 keys.  Per query tile TMEM holds ONE score buffer S and TWO
//   P buffers: a softmax thread pulls its S_j row into registers and releases the buffer at once (s_free), so
//   QK_{j+1} runs under the exponentials of step j; P_j goes to its own buffer, so PV_j never blocks a QK.
//   Inside a softmax warp the step is software-pipelined: the load of S_{j+1} and its row maximum are
//   interleaved with the last exponentials of step j, so a warp issues MUFU work almost without gaps.  That
//   matters because at D = 128 the exp unit (MUFU, 16 / clk / SM), not the tensor pipe, bounds FP8 attention.
//   To go past that bound a compile-time fraction of the exponentials is evaluated on the FMA pipe
//   (Cody-Waite split + minimax polynomial, packed fp32x2 arithmetic) instead of MUFU.EX2.
//   TMEM (512 columns): S_t at t*128 | P(t,b) at t*128 + 64 + b*32 | L_t at t*128 + 80 (row sums of P, single-e4m3
//   mode) | O_t at 256 + t*128.
//   K and V tiles are shared by both query tiles, halving L2->SMEM traffic per FLOP.
//
// Deliberately absent: any non-sm_100 path, any fallback.
#pragma once
#include <cmath>
#include <type_traits>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "ptx.cuh"
#include "qattn_internal.h"
#include "tma_host.h"

namespace qa {

#ifdef QA_TRACE
extern long long* g_trace_ptr;
extern int g_trace_x, g_trace_y;
#define QA_STAMP(role, step, ev)                                                                   \
    do {                                                                                          \
        if (p.trace && blockIdx.x == p.trace_x && blockIdx.y == p.trace_y && blockIdx.z == 0 && lane == 0 && (step) < 80) \
            p.trace[((role) * 80 + (step)) * 8 + (ev)] = clock64();                               \
    } while (0)
#else
#define QA_STAMP(role, step, ev) do { } while (0)
#endif

constexpr int BM = 128;  // query rows per tile (= TMEM lanes)
constexpr int BN = 128;  // keys per K/V shared-memory tile (one TMA box)
constexpr int BS = 64;   // keys per softmax / MMA step (half a tile)
constexpr float kLog2e = 1.4426950408889634f;
constexpr int kTmemCols = 512;  // one CTA per SM owns all of tensor memory
// setmaxnreg moves registers inside the allocation the CTA was launched with (two query tiles: 12 warps x 168 =
// 8 softmax warps x 224 + 4 MMA / TMA warps x 56)
constexpr int kRegSoftmax = 224, kRegOther = 56;

#ifndef QA_SYNCCHECK
#define QA_SYNCCHECK 0  // 1: the softmax threads wait for EVERY PV_{j-1} (compute-sanitizer synccheck flags barrier phases nobody
                        // observed; the shipping kernel only waits for a PV where its completion matters - rescale, last step)
#endif

// QK16_: Q and K stay 16-bit (bf16 / fp16) and QK^T runs as kind::f16 - the reference's `attn_func` path
// (src/quantum_attn/tk/attention.py:238-240,289-313); it implies the 16-bit P mode and has no dequantisation scales.
// PF16_: the 16-bit type of P (= V = out) in the 16-bit P mode is fp16 (else bf16).  A compile-time choice: selected at run
// time, the compiler converts every pair of probabilities to BOTH formats and picks one (64 extra F2FP per two steps
// and thread in the round-2 stall table: 9 % of the softmax loop's instructions).
template <int D_, int PMODE_, bool QK16_ = false, bool PF16_ = false>
struct AttnCfg {
    static constexpr int D = D_;
    static constexpr int PMODE = PMODE_;
    static constexpr bool QK16 = QK16_;
    static constexpr bool PF16 = PF16_;
    static constexpr bool V16 = (PMODE_ == QA_P_16BIT);
    static_assert(!QK16_ || V16, "16-bit Q/K go with 16-bit P and V");
    // query tiles per CTA: two share the K / V tiles of one CTA, but O for two tiles does not fit TMEM at D = 256
    static constexpr int NQ = D_ <= 128 ? 2 : 1;
    // Q in TENSOR MEMORY (D = 256).  An SS-form tcgen05.mma (A and B from shared memory) first loads its A operand - 128
    // rows x 32 bytes - which costs ~43 cycles per MMA on top of the N / 2 cycles of the product itself: measured on
    // B200 (scripts/ubench/mma_rate.cu) M128 x N64 x K32 takes 75 cycles from shared memory and 42 with A in TMEM.  Q
    // never changes during a tile, so the softmax threads put their query row into TMEM once (thread r = lane r, D
    // bytes = D / 4 columns, straight from global memory) and Q K^T runs as a TS-form MMA like P V does.  At D = 256 a
    // CTA holds ONE query tile, its 8 + 4 MMAs per step bound the step, and the TMEM columns are there: 633 -> 600 us
    // (16-bit P) / 510 -> 477 us (e4m3 P) on B16 S8192, causal 316 -> 289 us.  At D <= 128 the two tiles of a CTA
    // leave no columns for Q unless P goes down to one buffer, and there the tensor pipe is not what bounds the step:
    // measured SLOWER with Q in TMEM (C2 168.6 -> 184.8 us; one P buffer alone 172.4 -> 180.6 us), so those shapes
    // keep Q in shared memory.  Not for 16-bit Q.
    static constexpr bool QTMEM = D_ == 256 && !QK16_;
    static constexpr bool REBALANCE = NQ == 2;  // setmaxnreg: registers move to the softmax warps
    static constexpr int VB = V16 ? 2 : 1;          // bytes per V element
    static constexpr int QB = QK16_ ? 2 : 1;        // bytes per Q / K element
    // shared-memory tiles are stored as "boxes" whose rows are one swizzle span (<= 128 bytes) wide
    static constexpr int QK_ROW = (D_ * QB) < 128 ? (D_ * QB) : 128;  // bytes per box row for Q / K
    static constexpr int QK_BOXES = D_ * QB / QK_ROW;
    static constexpr int QK_BOX_BYTES = QK_ROW * 128;
    static constexpr int V_ROW = (D_ * VB) < 128 ? (D_ * VB) : 128;
    static constexpr int V_BOXES = D_ * VB / V_ROW;
    static constexpr int V_BOX_BYTES = V_ROW * BN;
    static constexpr int Q_TILE = QTMEM ? 0 : BM * D_ * QB;
    static constexpr int K_TILE = BN * D_ * QB;
    static constexpr int V_TILE = BN * D_ * VB;
    static constexpr int STAGES = QK16_ ? (D_ == 64 ? 4 : (D_ == 128 ? 2 : 1)) : (D_ == 64 ? 4 : (D_ == 128 ? 3 : 2));
    static constexpr int SMEM_Q = 0;
    static constexpr int SMEM_K = SMEM_Q + NQ * Q_TILE;
    static constexpr int SMEM_V = SMEM_K + STAGES * K_TILE;
    // single-e4m3 P mode: the row sums of P are accumulated by the tensor core, L (+)= P . 1, with a constant tile of
    // e4m3 ones (0x38) as the B operand - every byte the MMA can touch holds the same value, so the tile's layout is
    // immaterial - and a 16-column accumulator per query tile in the TMEM columns the 16-bit P buffers leave unused.
    // Not at D = 256, where the extra MMA costs more than the FADDs it saves (DESIGN.md section 4.2).
    static constexpr bool MMASUM = PMODE_ == QA_P_E4M3 && !QK16_ && D_ != 256;
    static constexpr int ONES_BYTES = MMASUM ? 4096 : 0;  // 32 keys x one swizzle span
    static constexpr int SMEM_ONES = SMEM_V + STAGES * V_TILE;
    static constexpr int SMEM_BAR = SMEM_ONES + ONES_BYTES;  // struct Barriers, 512 bytes reserved
    // per-token K scales (token-wise kernels): the 128 scales of a K / V tile ride the V ring - one 512-byte bulk copy
    // per tile next to the V boxes, completing on the same barrier - and the softmax threads read them from shared memory
    static constexpr int SMEM_SK = SMEM_BAR + 512;
    static constexpr int SK_BYTES = STAGES * BN * 4;
    static constexpr int SMEM_TOTAL = SMEM_SK + SK_BYTES + 1024;  // + alignment slack
    static_assert(SMEM_TOTAL + 1024 <= 233472, "shared memory budget exceeded");
    static constexpr int NSOFT = NQ * 4;                // softmax warps
    static constexpr int NTHREADS = (NSOFT + 4) * 32;   // softmax warpgroups + one warpgroup holding the MMA / TMA warps
    // TMEM columns
    static constexpr int TM_S = 0;                        // S_t at t * 128 (64 columns)
    static constexpr int TM_P = 64;                       // P(t, b) at t * 128 + 64 + b * 32
    static constexpr int TM_O = 256;                      // O_t at 256 + t * 128 (D <= 128), single O at D = 256
    static constexpr int TM_P_LO = 16;                    // hi/lo mode: second P tile 16 columns after the first
    static constexpr int TM_L = 80;                       // MMASUM: L_t at t * 128 + 80 (16 columns, column 0 is read)
    static constexpr int TM_Q = 128;                      // QTMEM (D = 256, one tile): Q in the D / 4 columns after P

    // softmax range management: p' = 2^KOFF * exp2(s - m_used), m_used may lag the true max by <= TAU (log2 units)
    static constexpr float KOFF = V16 ? 0.f : 4.f;
    static constexpr float TAU = V16 ? 8.f : 4.f;
    // Exponentials on the FMA pipe: of every 8 pairs, POLY_NUM are evaluated as a polynomial instead of by MUFU.EX2.
    // The share is a per-head-dimension balance, measured with scripts/time_shape.py: at D = 64 the MUFU is the contended
    // unit (little tensor work per score), at D = 256 a CTA has one softmax warp per scheduler, the MUFU is never
    // contended and every polynomial is pure extra issue work.  3 of 8 where the tensor core sums the rows (D = 64 and
    // 128 with a single e4m3 P), 2 of 8 elsewhere (16-bit P mode, C2 kernel 177.8 / 173.0 / 167.7 / 173.0 / 175.5 us at
    // 0..4 of 8).  Polynomial degree: a single e4m3 P tolerates the quadratic's 1.7e-3.
    static constexpr int POLY_NUM = MMASUM ? 3 : 2;
    static constexpr int POLY_DEG = (PMODE_ == QA_P_E4M3) ? 2 : 3;
};

struct AttnParams {
    const float* scale_q;
    const float* scale_k;
    const float* scale_v;
    float* lse;
    void* out;  // dense [B, Hq, Sq, D], 16 bit
    const uint8_t* q;            // QTMEM: e4m3 Q and its (batch, head, row) strides in bytes
    long long q_sb, q_sh, q_sr;
    int B, Hq, Hkv, Sq, Skv;
    int causal;
    int off;  // causal diagonal offset (>= 0): row i sees keys j <= i + off (0: top-left, Skv - Sq: bottom-right)
    float sm_scale_log2;  // sm_scale * log2(e)
    int out_fp16;
    int qk_fp16;  // QK16 configs: element type of Q and K
    int sk_bulk;  // token-wise: rows of scale_k are 16-byte aligned -> staged through shared memory by bulk copies
    // gated launch (qa_fp8_attn_fwd_gated): K / V of kv head h are only read once the `gate_flags` words from
    // kv_ready[(h / gate_heads) * gate_flags] on are all non-zero (set in stream order behind the copies that bring them)
    const unsigned* kv_ready;
    int gate_heads, gate_flags;
    float inv_group;  // Hkv / Hq
    long long* trace;  // developer builds (-DQA_TRACE): per-step clock64 stamps of one CTA, else unused
    int trace_x, trace_y;
};

struct Barriers {
    uint64_t q_full[2];
    uint64_t k_full[4], k_empty[4], v_full[4], v_empty[4];
    uint64_t s_full[2], s_free[2];  // [tile]: S_j written by the tensor core / pulled into registers by the softmax
    uint64_t p_full[2][2];          // [tile][P buffer]
    uint64_t pv_done[2][2], o_full[2];  // pv_done[tile][step parity]: PV_j complete
    uint32_t tmem_base;
};
static_assert(sizeof(Barriers) <= 512, "barrier block too large");

template <class C>
__device__ __forceinline__ uint32_t qk_koff(int k) {  // byte offset of the k-th 32-byte K slice inside a Q/K tile
    constexpr int per_box = C::QK_ROW / 32;
    return uint32_t(k / per_box) * C::QK_BOX_BYTES + uint32_t(k % per_box) * 32u;
}

// ------------------------------------------------------------------------------------------------ exp2 helpers
// 2^x for a pair of arguments on the FMA / ALU pipes: x = n + f with n = round(x) taken from the low mantissa bits of
// x + 1.5 * 2^23, f in [-0.5, 0.5], 2^f by a minimax polynomial (relative error 1.7e-3 / 7.5e-5 for degree 2 / 3),
// and n added straight into the exponent field.  Arguments are clamped at -125 (result ~ 2^-125, i.e. zero).
template <int DEG>
__device__ __forceinline__ float2 exp2_poly(float2 x) {
    x.x = fmaxf(x.x, -125.f);
    x.y = fmaxf(x.y, -125.f);
    const float2 magic = make_float2(12582912.f, 12582912.f);
    const float2 t = __fadd2_rn(x, magic);
    const float2 n = __fadd2_rn(t, make_float2(-12582912.f, -12582912.f));
    const float2 f = __ffma2_rn(n, make_float2(-1.f, -1.f), x);
    float2 q;
    if constexpr (DEG == 2) {
        q = __ffma2_rn(f, make_float2(0.23842893540859222f, 0.23842893540859222f),
                       make_float2(0.7034479975700378f, 0.7034479975700378f));
        q = __ffma2_rn(q, f, make_float2(1.0004431009292603f, 1.0004431009292603f));
    } else {
        q = __ffma2_rn(f, make_float2(0.0551716685295105f, 0.0551716685295105f),
                       make_float2(0.2426111251115799f, 0.2426111251115799f));
        q = __ffma2_rn(q, f, make_float2(0.6932609677314758f, 0.6932609677314758f));
        q = __ffma2_rn(q, f, make_float2(0.9999280571937561f, 0.9999280571937561f));
    }
    float2 r;
    r.x = __int_as_float(__float_as_int(q.x) + (__float_as_int(t.x) << 23));
    r.y = __int_as_float(__float_as_int(q.y) + (__float_as_int(t.y) << 23));
    return r;
}

__host__ __device__ constexpr bool pair_uses_poly(int i, int num) {  // spread `num` of every 8 pairs evenly
    return (((i & 7) + 1) * num) / 8 > ((i & 7) * num) / 8;
}

template <class C, bool CAUSAL, bool TOKEN>
__global__ void __launch_bounds__(C::NTHREADS, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, AttnParams p) {
    constexpr int D = C::D;
    constexpr int NQ = C::NQ;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    Barriers* bars = reinterpret_cast<Barriers*>(smem + C::SMEM_BAR);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int h = blockIdx.y, b = blockIdx.z;
    const int hkv = int((float(h) + 0.5f) * p.inv_group);  // exact for h < 2^16; avoids an integer-division call
    const int bh = b * p.Hq + h;
    const int bhkv = b * p.Hkv + hkv;
    // heavy (late) causal query blocks are scheduled first
    const int mblk = CAUSAL ? (gridDim.x - 1 - blockIdx.x) : blockIdx.x;
    const int m0 = mblk * (BM * NQ);
    const int nst_all = (p.Skv + BS - 1) / BS;
    // per-tile trip counts in 64-key steps: under a causal mask tile t stops at the step holding its last row's last
    // visible key, off + m0 + t * BM + BM - 1.  The producer (n_kv), the MMA warps and the softmax warps all take their
    // counts from n_steps(): a count that differed between the roles would leave a barrier waiting for ever
    const int nst0 = CAUSAL ? min(nst_all, (p.off + m0 + BM - 1) / BS + 1) : nst_all;
    const int nst1 = CAUSAL ? min(nst_all, (p.off + m0 + 2 * BM - 1) / BS + 1) : nst_all;
    auto n_steps = [&](int t) { return t == 0 ? nst0 : nst1; };
    const int n_max = n_steps(NQ - 1);
    const int n_kv = (n_max + 1) >> 1;  // K/V tiles of 128 keys

    QA_STAMP(warp >> 2, 78, 0);
    // the next kernel of the stream (typically the quantiser of the next call) may be scheduled as SMs drain
    griddep_launch_dependents();
    // ------------------------------------------------------------------ one-time setup
    // (everything up to the griddep_wait()s below touches no global data: it overlaps the tail of the previous kernel,
    // normally the quantiser that produces q8 / k8 / v8 and their scales)
    if (warp == 0) {
        tmem_alloc(&bars->tmem_base, kTmemCols);
        tmem_relinquish();
    }
    if (warp == 1) {  // one barrier per lane
        if (lane < 4) {
            const int t = lane >> 1, x = lane & 1;
            if (x) mbar_init(&bars->o_full[t], 1);
            mbar_init(&bars->pv_done[t][x], 1);
            mbar_init(&bars->p_full[t][x], BM);  // (s_free, p_full: every softmax thread of the tile arrives)
            mbar_init(x ? &bars->s_free[t] : &bars->s_full[t], x ? BM : 1);
        }
        fence_barrier_init();
    }
    // The TMA producer initialises its own barriers and starts Q and the first K / V tiles right away: their flight
    // time (about as long as the rest of the setup - TMEM allocation, the CTA-wide barrier) is then off the critical path.
    const int n_pre = min(n_kv, C::STAGES);
    auto load_kv = [&](int n) {
        const int s = n % C::STAGES;
        mbar_arrive_expect_tx(&bars->k_full[s], C::K_TILE);
        for (int x = 0; x < C::QK_BOXES; ++x)
            tma_load_4d(smem + C::SMEM_K + s * C::K_TILE + x * C::QK_BOX_BYTES, &tmK, &bars->k_full[s],
                        x * (C::QK_ROW / C::QB), n * BN, hkv, b, kEvictLast);
    };
    auto load_v = [&](int n) {
        const int s = n % C::STAGES;
        if constexpr (TOKEN) {
            if (p.sk_bulk) {  // the tile's per-token K scales land with its V boxes (a ragged tail copies what exists)
                const uint32_t sk_bytes = uint32_t(min(BN, p.Skv - n * BN)) * 4u;
                mbar_arrive_expect_tx(&bars->v_full[s], C::V_TILE + sk_bytes);
                bulk_load_1d(smem + C::SMEM_SK + s * (BN * 4), p.scale_k + size_t(bhkv) * p.Skv + size_t(n) * BN, sk_bytes,
                             &bars->v_full[s], kEvictLast);
            } else {
                // rows of scale_k not 16-byte aligned (Skv % 4 != 0): no bulk copy - the whole producer warp moves the 128
                // scales with plain loads (load_sk_warp) and arrives a second time: the barrier counts two arrivals per phase
                mbar_arrive_expect_tx(&bars->v_full[s], C::V_TILE);
            }
        } else {
            mbar_arrive_expect_tx(&bars->v_full[s], C::V_TILE);
        }
        for (int x = 0; x < C::V_BOXES; ++x)
            tma_load_4d(smem + C::SMEM_V + s * C::V_TILE + x * C::V_BOX_BYTES, &tmV, &bars->v_full[s],
                        x * (C::V_ROW / C::VB), n * BN, hkv, b, kEvictLast);
    };
    auto load_sk_warp = [&](int n) {  // (whole warp, converged; slot `s` is known to be free)
        const int s = n % C::STAGES;
        const float* src = p.scale_k + size_t(bhkv) * p.Skv;
        float a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] = __ldg(src + min(n * BN + lane * 4 + u, p.Skv - 1));
        reinterpret_cast<float4*>(smem + C::SMEM_SK + s * (BN * 4))[lane] = make_float4(a[0], a[1], a[2], a[3]);
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->v_full[s]);
    };
    if (warp == C::NSOFT + 1) {
        if (lane < 4) {
            mbar_init(&bars->k_full[lane], 1);
            mbar_init(&bars->k_empty[lane], NQ);  // released by every tile's MMA warp
            mbar_init(&bars->v_full[lane], (TOKEN && !p.sk_bulk) ? 2 : 1);
            mbar_init(&bars->v_empty[lane], NQ);
        } else if (lane < 4 + NQ) {
            mbar_init(&bars->q_full[lane - 4], C::QTMEM ? BM : 1);  // QTMEM: the tile's 128 rows, each put there by its thread
        }
        fence_barrier_init();
        __syncwarp();
        if (lane == 0) {
            tma_prefetch_desc(&tmQ);
            tma_prefetch_desc(&tmK);
            tma_prefetch_desc(&tmV);
            griddep_wait();
            if (p.kv_ready != nullptr) {
                // gated launch: this head's K / V may still be on their way (copy engines, another stream).  A bounded
                // poll: a transfer that never completes becomes a trap, not a hang.
                const unsigned* f = p.kv_ready + (hkv / p.gate_heads) * p.gate_flags;
                for (int i = 0; i < p.gate_flags; ++i) {
                    unsigned spins = 0;
                    while (ld_acquire_sys_u32(f + i) == 0u) {
                        __nanosleep(128);
                        if (++spins > (1u << 25)) __trap();
                    }
                }
                fence_proxy_async_global();  // the TMA engine (async proxy) reads what the flags vouch for
            }
            if constexpr (C::QTMEM) {
                load_kv(0);
            } else {
                for (int t = 0; t < NQ; ++t) {
                    mbar_arrive_expect_tx(&bars->q_full[t], C::Q_TILE);
                    for (int x = 0; x < C::QK_BOXES; ++x)
                        tma_load_4d(smem + C::SMEM_Q + t * C::Q_TILE + x * C::QK_BOX_BYTES, &tmQ, &bars->q_full[t],
                                    x * (C::QK_ROW / C::QB), m0 + t * BM, h, b, kEvictFirst);
                    if (t == 0) load_kv(0);  // K tile 0 right behind the first Q tile: S_0 needs exactly these two
                }
            }
            load_v(0);
            for (int n = 1; n < n_pre; ++n) {
                load_kv(n);
                load_v(n);
            }
        }
        if constexpr (TOKEN) {
            if (!p.sk_bulk) {
                griddep_wait();  // (every lane reads scale_k, which the quantiser of this call wrote)
                __syncwarp();
                for (int n = 0; n < n_pre; ++n) load_sk_warp(n);
            }
        }
    }
    if constexpr (C::MMASUM) {
        for (int i = threadIdx.x; i < C::ONES_BYTES / 4; i += C::NTHREADS)
            reinterpret_cast<uint32_t*>(smem + C::SMEM_ONES)[i] = 0x38383838u;  // e4m3 1.0
        fence_proxy_async_smem();  // the tensor core reads shared memory through the async proxy
    }
    griddep_wait();  // (the TMA lane has passed its own wait already: a second one returns at once)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // the CTA owns all 512 columns, so the allocation starts at column 0: TMEM addresses are the TM_* offsets below
    if (bars->tmem_base != 0) __trap();

    // register rebalancing (two-tile configs run 384 threads -> 168 registers each at launch): the softmax
    // warpgroups keep a whole score row per thread in registers, the MMA / TMA warps need almost nothing
    if (warp >= C::NSOFT) {
        if constexpr (C::REBALANCE) reg_dealloc<kRegOther>();
        if (warp == C::NSOFT + 1) {
            // =========================================================== TMA producer
            if (TOKEN && !p.sk_bulk) {
                // (unaligned per-token K scales: lane 0 runs the ring as below, the whole warp then fills the scale slot)
                for (int n = n_pre; n < n_kv; ++n) {
                    const int s = n % C::STAGES;
                    const uint32_t ph = (n / C::STAGES) & 1;
                    if (lane == 0) {
                        mbar_wait(&bars->k_empty[s], ph ^ 1);
                        load_kv(n);
                        mbar_wait(&bars->v_empty[s], ph ^ 1);
                        load_v(n);
                    }
                    __syncwarp();
                    load_sk_warp(n);
                }
            } else if (lane == 0) {
                for (int n = n_pre; n < n_kv; ++n) {  // (Q and the first n_pre tiles were issued during the setup)
                    const int s = n % C::STAGES;
                    const uint32_t ph = (n / C::STAGES) & 1;
                    mbar_wait(&bars->k_empty[s], ph ^ 1);
                    load_kv(n);
                    mbar_wait(&bars->v_empty[s], ph ^ 1);
                    load_v(n);
                }
            }
        } else if (warp == C::NSOFT || (NQ == 2 && warp == C::NSOFT + 2)) {
            // =========================================================== MMA issuers: one warp per query tile
            // Each tile has its own chain  P_j -> PV_j -> QK_{j+2} -> S_{j+2}; a warp per tile keeps the two chains
            // independent (a single in-order issuer would couple them) and halves the per-step instruction stream.
            // The warp walks the loop converged; one elected lane issues.  Descriptors are built once: per MMA only
            // the 14-bit start-address field of the low word changes.
            const int t = (warp - C::NSOFT) >> 1;
            const int nst = n_steps(t);
            const uint32_t qk_fmt = (C::QK16 && !p.qk_fp16) ? 1u : 0u;  // f16: 0 = fp16, 1 = bf16;  f8f6f4: 0 = e4m3
            const uint32_t idesc_qk = make_idesc(qk_fmt, qk_fmt, 0, 0, BM, BS);
            constexpr uint32_t idesc_pv8 = make_idesc(0, 0, 0, 1, BM, D);
            const uint32_t idesc_pv = C::V16 ? make_idesc(C::PF16 ? 0 : 1, C::PF16 ? 0 : 1, 0, 1, BM, D) : idesc_pv8;
            constexpr uint64_t qk_swz = (C::QK_ROW == 128) ? kSwz128 : kSwz64;
            constexpr uint64_t v_swz = (C::V_ROW == 128) ? kSwz128 : kSwz64;
            const uint64_t q_desc = make_smem_desc(smem_u32(smem + C::SMEM_Q + t * C::Q_TILE), 16, 8 * C::QK_ROW, qk_swz);
            const uint64_t k_desc0 = make_smem_desc(smem_u32(smem + C::SMEM_K), 16, 8 * C::QK_ROW, qk_swz);
            const uint64_t v_desc0 = make_smem_desc(smem_u32(smem + C::SMEM_V), C::V_BOX_BYTES, 8 * C::V_ROW, v_swz);
            constexpr int KEYS_PER_PV = C::V16 ? 16 : 32;
            const uint32_t s_t = C::TM_S + t * 128;
            const uint32_t p_t0 = C::TM_P + t * 128;
            const uint32_t q_t = C::TM_Q + t * 128;  // QTMEM: K slice k of Q_t = 8 columns at q_t + 8 k
            const uint32_t o_t = C::TM_O + (NQ == 2 ? t * 128 : 0);
            const uint32_t l_t = C::TM_L + t * 128;
            constexpr uint32_t idesc_l = make_idesc(0, 0, 0, 1, BM, 16);
            const uint64_t ones_desc = make_smem_desc(smem_u32(smem + C::SMEM_ONES), C::V_BOX_BYTES, 8 * C::V_ROW, v_swz);

            // S_t = Q_t . K[64 keys]^T, the keys being rows [half * 64, half * 64 + 64) of K stage `stage`
            auto issue_qk = [&](int stage, int half) {
                const uint64_t bd = k_desc0 + uint64_t((stage * C::K_TILE + half * (BS * C::QK_ROW)) >> 4);
#pragma unroll
                for (int k = 0; k < D * C::QB / 32; ++k) {  // one MMA per 32-byte K slice (32 e4m3 / 16 bf16 elements)
                    if constexpr (C::QK16)
                        umma_f16_ss(s_t, q_desc + (qk_koff<C>(k) >> 4), bd + (qk_koff<C>(k) >> 4), idesc_qk, k > 0);
                    else if constexpr (C::QTMEM)
                        umma_f8_ts(s_t, q_t + k * 8, bd + (qk_koff<C>(k) >> 4), idesc_qk, k > 0);
                    else
                        umma_f8_ss(s_t, q_desc + (qk_koff<C>(k) >> 4), bd + (qk_koff<C>(k) >> 4), idesc_qk, k > 0);
                }
            };
            // O_t (+)= P(t, half) . V[64 keys]
            auto issue_pv = [&](int stage, int half, bool acc) {
                const uint32_t p_t = p_t0 + half * 32;
                const uint64_t bd = v_desc0 + uint64_t((stage * C::V_TILE + half * (BS * C::V_ROW)) >> 4);
#pragma unroll
                for (int k = 0; k < BS / KEYS_PER_PV; ++k) {
                    const uint64_t bk = bd + uint64_t((k * KEYS_PER_PV * C::V_ROW) >> 4);
                    if constexpr (!C::V16) {
                        umma_f8_ts(o_t, p_t + k * 8, bk, idesc_pv, (acc || k > 0) ? 1u : 0u);
                        if constexpr (C::PMODE == QA_P_E4M3_HILO) umma_f8_ts(o_t, p_t + C::TM_P_LO + k * 8, bk, idesc_pv, 1u);
                        if constexpr (C::MMASUM) umma_f8_ts(l_t, p_t + k * 8, ones_desc, idesc_l, (acc || k > 0) ? 1u : 0u);
                    } else {
                        umma_f16_ts(o_t, p_t + k * 8, bk, idesc_pv, (acc || k > 0) ? 1u : 0u);
                    }
                }
            };

            // prologue: S_0 and (once S_0 has been pulled) S_1 from K tile 0
            mbar_wait(&bars->q_full[t], 0);
            mbar_wait(&bars->k_full[0], 0);
            tc_fence_after();
            if (elect_one()) {
                issue_qk(0, 0);
                umma_commit(&bars->s_full[t]);
                if (nst == 1) umma_commit(&bars->k_empty[0]);
            }
            __syncwarp();
            if (nst > 1) {
                mbar_wait(&bars->s_free[t], 0);
                tc_fence_after();
                if (elect_one()) {
                    issue_qk(0, 1);
                    umma_commit(&bars->s_full[t]);
                    umma_commit(&bars->k_empty[0]);
                }
                __syncwarp();
            }

            // steady state, one K/V tile (two steps) per trip; the score GEMM runs two steps ahead of the PV GEMM:
            //   [s_free(j+1) -> QK_{j+2}]  [p_full(j) -> PV_j]  [s_free(j+2) -> QK_{j+3}]  [p_full(j+1) -> PV_{j+1}]
            int sv = 0, sk = 0;       // ring slots of the V tile feeding PV_j and of the K tile feeding QK_{j+2}
            uint32_t pv = 0, pk = 0;  // their parities
            uint32_t pp = 0;          // parity of p_full[t][*] (both buffers flip once per trip)
            for (int j = 0; j < nst; j += 2) {
                const bool has1 = j + 1 < nst, has2 = j + 2 < nst, has3 = j + 3 < nst;
                if (++sk == C::STAGES) sk = 0, pk ^= 1;
                if (has2) {
                    // ---- QK_{j+2}: first half of the next K tile
                    mbar_wait(&bars->k_full[sk], pk);
                    mbar_wait(&bars->s_free[t], 1);
                    tc_fence_after();
                    if (elect_one()) {
                        issue_qk(sk, 0);
                        umma_commit(&bars->s_full[t]);
                        if (!has3) umma_commit(&bars->k_empty[sk]);
                    }
                    __syncwarp();
                }
                QA_STAMP(2 + t, j, 0);
                // ---- PV_j: P buffer 0, first half of the V tile
                mbar_wait(&bars->v_full[sv], pv);
                mbar_wait(&bars->p_full[t][0], pp);
                tc_fence_after();
                QA_STAMP(2 + t, j, 1);
                if (elect_one()) {
                    issue_pv(sv, 0, j > 0);
                    umma_commit(&bars->pv_done[t][0]);
                    if (!has1) umma_commit(&bars->v_empty[sv]);
                }
                __syncwarp();
                QA_STAMP(2 + t, j, 2);
                if (has3) {
                    // ---- QK_{j+3}: second half of that K tile
                    mbar_wait(&bars->s_free[t], 0);
                    tc_fence_after();
                    if (elect_one()) {
                        issue_qk(sk, 1);
                        umma_commit(&bars->s_full[t]);
                        umma_commit(&bars->k_empty[sk]);
                    }
                    __syncwarp();
                }
                if (has1) {
                    QA_STAMP(2 + t, j + 1, 0);
                    // ---- PV_{j+1}: P buffer 1, second half of the V tile
                    mbar_wait(&bars->p_full[t][1], pp);
                    tc_fence_after();
                    QA_STAMP(2 + t, j + 1, 1);
                    if (elect_one()) {
                        issue_pv(sv, 1, true);
                        umma_commit(&bars->pv_done[t][1]);
                        umma_commit(&bars->v_empty[sv]);
                    }
                    __syncwarp();
                    QA_STAMP(2 + t, j + 1, 2);
                }
                pp ^= 1;
                if (++sv == C::STAGES) sv = 0, pv ^= 1;
            }
            if (elect_one()) umma_commit(&bars->o_full[t]);
            __syncwarp();
        }
    } else {
        // =============================================================== softmax / correction / epilogue
        if constexpr (C::REBALANCE) reg_alloc<kRegSoftmax>();
        const int t = warp / 4;                        // query tile of this warpgroup
        const int row = ((warp & 3) << 5) | lane;      // row inside the tile == TMEM lane
        const uint32_t lane_base = uint32_t((warp & 3) * 32) << 16;
        const uint32_t s_addr = lane_base + C::TM_S + t * 128;
        const uint32_t p_base = lane_base + C::TM_P + t * 128;
        const uint32_t o_addr = lane_base + C::TM_O + (NQ == 2 ? t * 128 : 0);
        const uint32_t l_addr = lane_base + C::TM_L + t * 128;
        const int row_g = m0 + t * BM + row;
        const int diag_t = CAUSAL ? p.off + m0 + t * BM : 0;  // last key the tile's first row sees (causal)

        float c;  // multiplier taking raw fp8 dot products to the base-2 softmax domain
        if constexpr (C::QK16) {
            c = p.sm_scale_log2;
        } else if constexpr (TOKEN) {
            c = p.scale_q[size_t(bh) * p.Sq + min(row_g, p.Sq - 1)] * p.sm_scale_log2;
        } else {
            c = p.scale_q[bh] * p.scale_k[bhkv] * p.sm_scale_log2;
        }
        const float2 c2 = make_float2(c, c);

        float m_used = -INFINITY;  // running max in raw score units (times per-column scale in token mode)
        float2 la = make_float2(0.f, 0.f), lb = make_float2(0.f, 0.f);  // running sum of p' (4 partial sums)
        const int my_steps = n_steps(t);

        // per-column K scales (token mode), applied to the raw scores of step j (called once per step, in order).  They
        // come from shared memory, where the producer put the tile's 128 scales with its V boxes: the slot is refilled
        // only after P V of the tile's second step, i.e. after every softmax thread has published that step's P.
        int sk_slot = 0;
        uint32_t sk_phase = 0;
        const uint32_t sk_base = smem_u32(smem + C::SMEM_SK);
        auto kscale = [&](const int j, float (&s)[BS]) {
            if constexpr (TOKEN) {
                if ((j & 1) == 0) {
                    if (j > 0 && ++sk_slot == C::STAGES) sk_slot = 0, sk_phase ^= 1;
                    mbar_wait(&bars->v_full[sk_slot], sk_phase);  // (long complete: V_n is loaded ahead of P V_2n)
                }
                const uint32_t sk_addr = sk_base + uint32_t(sk_slot * (BN * 4) + (j & 1) * (BS * 4));
#pragma unroll
                for (int i = 0; i < BS; i += 4) {
                    const float4 k4 = lds_f32x4(sk_addr + i * 4);
                    const float2 a = __fmul2_rn(make_float2(s[i], s[i + 1]), make_float2(k4.x, k4.y));
                    const float2 bq = __fmul2_rn(make_float2(s[i + 2], s[i + 3]), make_float2(k4.z, k4.w));
                    s[i] = a.x, s[i + 1] = a.y, s[i + 2] = bq.x, s[i + 3] = bq.y;
                }
            }
        };
        // causal / ragged mask of step j.  Only the trailing steps of a tile can need it (the ragged tail is the last
        // step, the causal diagonal the last two), so it is instantiated in the tail loop only: the main loop below
        // carries no mask code at all and stays a compact straight line for the instruction cache.
        auto mask = [&](const int j, float (&s)[BS]) {
            const int col0 = j * BS;
            const bool tail = col0 + BS > p.Skv;
            const bool diag = CAUSAL && (col0 + BS - 1 > diag_t);
            if (tail || diag) {
                const int lim = CAUSAL ? min(p.Skv - 1, diag_t + row) : (p.Skv - 1);  // last visible column
#pragma unroll
                for (int i = 0; i < BS; ++i)
                    if (col0 + i > lim) s[i] = -INFINITY;
            }
        };
        // first step whose scores need the mask (every later one does too)
        const int j_mask = CAUSAL ? min(p.Skv / BS, diag_t / BS) : p.Skv / BS;
        // row maximum of sixteen columns folded into two running maxima (two chains per call site -> four in flight)
        auto max16 = [&](const float (&s)[BS], int q, float& ma, float& mb) {
#pragma unroll
            for (int i = 16 * q; i < 16 * q + 16; i += 4) {
                ma = fmaxf(ma, fmaxf(s[i], s[i + 1]));
                mb = fmaxf(mb, fmaxf(s[i + 2], s[i + 3]));
            }
        };
        // rare: the running maximum of some row of this warp grew by more than 2^TAU -> rescale O (rolled: cold code)
        auto rescale_o = [&](const float alpha) {
#pragma unroll 1
            for (int cc = 0; cc < D; cc += 32) {
                float o[32];
                tmem_ld_x32(o_addr + cc, o);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; ++i) o[i] *= alpha;
                tmem_st_x32(o_addr + cc, o);
            }
            if constexpr (C::MMASUM) {  // the row sum lives beside O and is rescaled with it
                float lv = tmem_ld_x1(l_addr);
                tmem_ld_wait();
                tmem_st_x1(l_addr, lv * alpha);
            }
            tmem_st_wait();
        };

        // One 64-key step.  On entry `s` holds S_j (scaled / masked as needed) and `mx` its row maximum.  The step turns
        // S_j into P_j.  Unless it is the last step it also pulls S_{j+1} into `s_next` after LOADQ quads of
        // exponentials, frees the score buffer for QK_{j+2}, and folds the row maximum of S_{j+1} into the remaining
        // exponentials; it returns that maximum.  The code between the few waits is straight-line on purpose: every
        // branch is a scheduling barrier at which the exp pipeline of this warp drains.
        //   MASKED (compile time): S_{j+1} may need the causal / ragged mask;  `last`: there is no S_{j+1}.
        //   `need` (warp-uniform): some row of the warp has outgrown its stale maximum, as decided near the END of the
        //   previous step (see below) - so the common case enters the exponentials with nothing to wait for.
        auto step = [&](const int j, float (&s)[BS], float (&s_next)[BS], const float mx, bool& need, auto mask_tag,
                        const bool last) -> float {
            constexpr bool MASKED = decltype(mask_tag)::value;
            // The schedule of the step, in quads of exponentials (four columns each, NQD per step).  Each constant was
            // re-measured on the final kernel against its neighbours; none of those won on C2, C3 and D = 64 at once
            // (profiles/r02_tune_ab.txt).
            constexpr int NQD = BS / 4;
            constexpr int PUBQ = 2;     // P_{j-1} (stored at the end of step j-1) is published after this many quads
            constexpr int LOADQ = 8;    // S_{j+1} is pulled into registers after this many quads
            constexpr int LDWAITQ = 4;  // quads between the TMEM load of S_{j+1} and the wait for it
            constexpr int DECIDEQ = 1;  // quads left when the rescale decision for the next step is taken
            QA_STAMP(t, j, 0);
            bool p_prev_pending = j > 0;  // P_{j-1} is stored but not yet published (see below)
            // lazy rescale: keep the stale max while the true max has grown by < 2^TAU
            if (__builtin_expect(need, 0)) {
                const float m_new = fmaxf(m_used, mx);
                const float alpha = ex2_approx((m_used - m_new) * c);  // 0 on the first step
                m_used = m_new;
                if constexpr (!C::MMASUM) la.x *= alpha, la.y *= alpha, lb.x *= alpha, lb.y *= alpha;
                if (j > 0) {
                    // O_t must be quiescent: PV_{j-1} is the only MMA that can still be writing it - and it cannot
                    // even start before P_{j-1} is published
                    tmem_st_wait();
                    tc_fence_before();
                    mbar_arrive(&bars->p_full[t][(j - 1) & 1]);
                    p_prev_pending = false;
                    // (one barrier per step parity: PV_{j-3}, the previous phase of this barrier, is known to be
                    // complete because S_j has been seen, so the parity test cannot alias)
                    mbar_wait(&bars->pv_done[t][(j - 1) & 1], ((j - 1) >> 1) & 1);
                    tc_fence_after();
                    rescale_o(alpha);
                }
            }
            const float neg = C::KOFF - m_used * c;
            const float2 neg2 = make_float2(neg, neg);
            QA_STAMP(t, j, 1);

            // p' for one pair of columns; a compile-time subset of the pairs avoids MUFU
            auto exp_pair = [&](int i) -> float2 {
                const float2 x = __ffma2_rn(make_float2(s[2 * i], s[2 * i + 1]), c2, neg2);
                if (pair_uses_poly(i, C::POLY_NUM)) return exp2_poly<C::POLY_DEG>(x);
                return make_float2(ex2_approx(x.x), ex2_approx(x.y));
            };
            uint32_t pw[C::V16 ? BS / 2 : BS / 4], pw_lo[C::PMODE == QA_P_E4M3_HILO ? BS / 4 : 1];
            // four columns -> P words (and, unless the tensor core sums the rows of P, the running row sum)
            auto exp_quad = [&](int i) {
                const float2 p01 = exp_pair(2 * i), p23 = exp_pair(2 * i + 1);
                if constexpr (!C::MMASUM) {
                    la = __fadd2_rn(la, p01);
                    lb = __fadd2_rn(lb, p23);
                }
                if constexpr (C::PMODE == QA_P_E4M3) {
                    pw[i] = pack_e4m3x4(p01.x, p01.y, p23.x, p23.y);
                } else if constexpr (C::PMODE == QA_P_E4M3_HILO) {
                    const uint32_t h01 = cvt_e4m3x2(p01.x, p01.y), h23 = cvt_e4m3x2(p23.x, p23.y);
                    const float2 f01 = e4m3x2_to_float2(h01), f23 = e4m3x2_to_float2(h23);
                    pw[i] = h01 | (h23 << 16);
                    pw_lo[i] = pack_e4m3x4(p01.x - f01.x, p01.y - f01.y, p23.x - f23.x, p23.y - f23.y);
                } else {
                    pw[2 * i] = C::PF16 ? pack_f16x2(p01.x, p01.y) : pack_bf16x2(p01.x, p01.y);
                    pw[2 * i + 1] = C::PF16 ? pack_f16x2(p23.x, p23.y) : pack_bf16x2(p23.x, p23.y);
                }
            };

#pragma unroll
            for (int i = 0; i < PUBQ; ++i) exp_quad(i);
            if (p_prev_pending) {  // P_{j-1} was stored at the end of the previous step: publish it now
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(&bars->p_full[t][(j - 1) & 1]);
            }
#pragma unroll
            for (int i = PUBQ; i < LOADQ; ++i) exp_quad(i);
            float ma = -INFINITY, mb = -INFINITY;
            if (!last) {
                // S_{j+1} was issued by the tensor core when this thread released S_j, about one step ago
                QA_STAMP(t, j, 5);
                mbar_wait(&bars->s_full[t], (j + 1) & 1);
                tc_fence_after();
                tmem_ld_f64(s_addr, s_next);
                QA_STAMP(t, j, 2);
#pragma unroll
                for (int i = LOADQ; i < LOADQ + LDWAITQ; ++i) exp_quad(i);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(&bars->s_free[t]);  // the score buffer may be overwritten by QK_{j+2}
                kscale(j + 1, s_next);
                if constexpr (MASKED) mask(j + 1, s_next);
                QA_STAMP(t, j, 3);
                // the row maximum of S_{j+1} is spread over the remaining quads but the last DECIDEQ, four 16-column
                // pieces in all; the rescale decision for step j + 1 (a warp vote) is taken before those last quads, whose
                // exponentials hide its latency
                constexpr int REST = NQD - LDWAITQ - LOADQ - DECIDEQ;  // quads carrying a piece of the maximum
                static_assert(PUBQ <= LOADQ && REST >= 1, "quad schedule");
                constexpr int NPIECE = BS / 16;                  // 16-column pieces of the row maximum
                constexpr int PER = (NPIECE + REST - 1) / REST;  // pieces per quad
#pragma unroll
                for (int i = LOADQ + LDWAITQ; i < NQD - DECIDEQ; ++i) {
                    exp_quad(i);
#pragma unroll
                    for (int q = 0; q < PER; ++q) {
                        const int piece = (i - LOADQ - LDWAITQ) * PER + q;
                        if (piece < NPIECE) max16(s_next, piece, ma, mb);
                    }
                }
                need = __any_sync(0xffffffffu, (fmaxf(ma, mb) - m_used) * c > C::TAU);
#pragma unroll
                for (int i = NQD - DECIDEQ; i < NQD; ++i) exp_quad(i);
            } else {
                need = false;
#pragma unroll
                for (int i = LOADQ; i < NQD; ++i) exp_quad(i);
                // P buffer reuse: PV_{j-2} must have drained it.  Seeing S_{j+1} (issued after PV_{j-2}, in-order
                // tensor pipe) proves that in every other step; the last one waits for PV_{j-1} explicitly.
                if (j >= 2) mbar_wait(&bars->pv_done[t][(j - 1) & 1], ((j - 1) >> 1) & 1);
            }
            if constexpr (QA_SYNCCHECK != 0) {
                if (j >= 1 && !last) mbar_wait(&bars->pv_done[t][(j - 1) & 1], ((j - 1) >> 1) & 1);
            }
            // P_j goes to buffer j & 1 of the tile: 64 keys = 32 columns of 16-bit P or 16 columns of e4m3 P
            const uint32_t p_addr = p_base + (j & 1) * 32;
            if constexpr (C::PMODE == QA_P_E4M3) {
                tmem_st_words<BS / 4>(p_addr, pw);
            } else if constexpr (C::PMODE == QA_P_E4M3_HILO) {
                tmem_st_words<BS / 4>(p_addr, pw);
                tmem_st_words<BS / 4>(p_addr + C::TM_P_LO, pw_lo);
            } else {
                tmem_st_words<BS / 2>(p_addr, pw);
            }
            if (last) {  // nothing left to hide the store behind
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(&bars->p_full[t][j & 1]);
            }
            QA_STAMP(t, j, 4);
            return fmaxf(ma, mb);
        };

        if constexpr (C::QTMEM) {
            // this thread's query row -> tensor memory (lane = row, D bytes = D / 4 columns), straight from global
            // memory: the A operand of every Q K^T MMA of the tile
            const uint8_t* qrow = p.q + (long long)b * p.q_sb + (long long)h * p.q_sh +
                                  (long long)min(row_g, p.Sq - 1) * p.q_sr;
            const uint32_t q_addr = lane_base + C::TM_Q + t * 128;
            constexpr int NW = (D / 4 < 32) ? D / 4 : 32;  // words per tcgen05.st
#pragma unroll
            for (int c0 = 0; c0 < D / 4; c0 += NW) {
                uint32_t w[NW];
#pragma unroll
                for (int i = 0; i < NW; i += 4) {
                    const uint4 v = __ldg(reinterpret_cast<const uint4*>(qrow + (c0 + i) * 4));
                    w[i] = v.x, w[i + 1] = v.y, w[i + 2] = v.z, w[i + 3] = v.w;
                }
                tmem_st_words<NW>(q_addr + c0, w);
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(&bars->q_full[t]);
        }
        float s_a[BS], s_b[BS];
        float mx;
        QA_STAMP(t, 78, 1);
        {   // S_0
            mbar_wait(&bars->s_full[t], 0);
            QA_STAMP(t, 78, 2);
            tc_fence_after();
            tmem_ld_f64(s_addr, s_a);
            tmem_ld_wait();
            tc_fence_before();
            mbar_arrive(&bars->s_free[t]);
            kscale(0, s_a);
            mask(0, s_a);
            float ma = -INFINITY, mb = -INFINITY;
#pragma unroll
            for (int q = 0; q < BS / 16; ++q) max16(s_a, q, ma, mb);
            mx = fmaxf(ma, mb);
        }
        {
            using std::false_type;
            using std::true_type;
            // main loop: steps whose successor exists and needs no mask, two per trip (the score registers ping-pong)
            const int n_fast = min(my_steps - 1, j_mask - 1);
            int j = 0;
            bool need = true;  // first step: m_used = -inf
            for (; j + 2 <= n_fast; j += 2) {
                __builtin_assume((j & 1) == 0);  // (token-wise: the K-scale slot advances on even steps)
                mx = step(j, s_a, s_b, mx, need, false_type{}, false);
                mx = step(j + 1, s_b, s_a, mx, need, false_type{}, false);
            }
            // tail: the few steps around the causal diagonal / ragged end, and the last one (rolled, one instance; a
            // second, ping-pong pair of masked instances was measured: C3 404 -> 403 us in the default mode, 350 -> 361 us
            // with e4m3 P - the extra code costs more in the instruction cache than the register copy it saves)
#pragma unroll 1
            for (; j < my_steps; ++j) {
                mx = step(j, s_a, s_b, mx, need, true_type{}, j + 1 == my_steps);
#pragma unroll
                for (int i = 0; i < BS; ++i) s_a[i] = s_b[i];
            }
        }
        float l = (la.x + la.y) + (lb.x + lb.y);
        QA_STAMP(t, 78, 3);

        // ---------------------------------------------------------------- epilogue: O / l -> 16 bit -> global memory
        mbar_wait(&bars->o_full[t], 0);
        tc_fence_after();
        QA_STAMP(t, 78, 4);
        if constexpr (C::MMASUM) {
            l = tmem_ld_x1(l_addr);
            tmem_ld_wait();
        }
        const float sv = C::V16 ? 1.f : p.scale_v[bhkv];
        const float inv = __fdividef(sv, l);
        // A thread owns a whole output row (D * 2 contiguous bytes): it writes it straight from its registers, one
        // 32-byte sector per store.  Nothing to stage, fence or wait for - the CTA is free to retire as soon as the
        // stores are issued, where a shared-memory + TMA route would keep it alive until the bulk store had read the tile.
        uint8_t* o_row = static_cast<uint8_t*>(p.out) + (size_t(bh) * p.Sq + min(row_g, p.Sq - 1)) * (D * 2);
#pragma unroll
        for (int cc = 0; cc < D; cc += 32) {
            float o[32];
            tmem_ld_x32(o_addr + cc, o);
            tmem_ld_wait();
            uint32_t w[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float a = o[2 * i] * inv, bb = o[2 * i + 1] * inv;
                w[i] = p.out_fp16 ? pack_f16x2(a, bb) : pack_bf16x2(a, bb);
            }
            if (row_g < p.Sq) {
                st_global_32B(o_row + cc * 2, w);
                st_global_32B(o_row + cc * 2 + 32, w + 8);
            }
        }
        if (p.lse != nullptr && row_g < p.Sq)
            p.lse[size_t(bh) * p.Sq + row_g] = (m_used * c + (__log2f(l) - C::KOFF)) * 0.6931471805599453f;
        QA_STAMP(t, 78, 5);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(0, kTmemCols);
    QA_STAMP(warp >> 2, 78, 6);
}

// ------------------------------------------------------------------------------------------------ host side
template <class C, bool CAUSAL, bool TOKEN>
static int launch_cfg(const AttnArgs& a, cudaStream_t stream, int* launches) {
    CUtensorMap tmQ, tmK, tmV;
    const CUtensorMapSwizzle qk_swz = C::QK_ROW == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const CUtensorMapSwizzle v_swz = C::V_ROW == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const uint64_t D = C::D;
    bool ok = true;
    const CUtensorMapDataType qkdt = !C::QK16 ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                     : (a.qk_dtype == QA_DT_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                                 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
    // Q, K, V in place through their own batch / head / row strides (element strides in AttnArgs, D contiguous)
    ok &= make_tmap_4d(&tmQ, qkdt, a.q8, D, a.Sq, a.Hq, a.B, a.qs[2] * C::QB, a.qs[1] * C::QB, a.qs[0] * C::QB,
                       C::QK_ROW / C::QB, BM, qk_swz);
    ok &= make_tmap_4d(&tmK, qkdt, a.k8, D, a.Skv, a.Hkv, a.B, a.ks[2] * C::QB, a.ks[1] * C::QB, a.ks[0] * C::QB,
                       C::QK_ROW / C::QB, BN, qk_swz);
    {
        const CUtensorMapDataType dt = !C::V16 ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                       : (a.v_dtype == QA_DT_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                                  : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
        ok &= make_tmap_4d(&tmV, dt, a.v, D, a.Skv, a.Hkv, a.B, a.vs[2] * C::VB, a.vs[1] * C::VB, a.vs[0] * C::VB,
                           C::V_ROW / C::VB, BN, v_swz);
    }
    if (!ok) return set_error(QA_ERR_DEVICE, "cuTensorMapEncodeTiled failed or is unavailable (no CUDA driver?)");

    AttnParams p;
    p.scale_q = a.scale_q;
    p.scale_k = a.scale_k;
    p.scale_v = a.scale_v;
    p.lse = a.lse;
    p.out = a.out;
    p.q = static_cast<const uint8_t*>(a.q8);
    p.q_sb = a.qs[0] * C::QB, p.q_sh = a.qs[1] * C::QB, p.q_sr = a.qs[2] * C::QB;
    p.B = a.B, p.Hq = a.Hq, p.Hkv = a.Hkv, p.Sq = a.Sq, p.Skv = a.Skv;
    p.causal = a.causal;
    p.off = a.causal == QA_CAUSAL_BOTTOM_RIGHT ? a.Skv - a.Sq : 0;
    p.sm_scale_log2 = a.sm_scale * kLog2e;
    p.out_fp16 = (a.out_dtype == QA_DT_FP16);
    p.qk_fp16 = (a.qk_dtype == QA_DT_FP16);
    p.sk_bulk = TOKEN && (a.Skv % 4 == 0) && (reinterpret_cast<uintptr_t>(a.scale_k) % 16 == 0);
    p.kv_ready = a.kv_ready, p.gate_heads = a.gate_heads > 0 ? a.gate_heads : 1, p.gate_flags = a.gate_flags;
    p.inv_group = float(a.Hkv) / float(a.Hq);
#ifdef QA_TRACE
    p.trace = g_trace_ptr;
    p.trace_x = g_trace_x, p.trace_y = g_trace_y;
#else
    p.trace = nullptr;
    p.trace_x = p.trace_y = 0;
#endif

    auto kern = attn_fwd_kernel<C, CAUSAL, TOKEN>;
    static DeviceSet attr_done;  // per instantiation and per device (function attributes belong to a device)
    const int dev = current_device();
    if (!attr_done.has(dev)) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_TOTAL);
        if (e != cudaSuccess) return set_cuda_error("cudaFuncSetAttribute(max dynamic smem)", e);
        attr_done.add(dev);
    }
    dim3 grid((a.Sq + BM * C::NQ - 1) / (BM * C::NQ), a.Hq, a.B);
    cudaError_t e = launch_pdl(kern, grid, dim3(C::NTHREADS), size_t(C::SMEM_TOTAL), stream, tmQ, tmK, tmV, p);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error("attn_fwd_kernel launch", e);
    *launches += 1;
    return QA_OK;
}

}  // namespace qa
