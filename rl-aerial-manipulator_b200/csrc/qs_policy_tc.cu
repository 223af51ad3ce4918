// qs_policy_tc.cu -- MlpPolicy rollout forward on tcgen05 with the activations kept in TENSOR MEMORY (A operand from
// TMEM, "TS" form of tcgen05.mma) and, in PRECISE mode, split-float16 arithmetic that reproduces float32 accuracy.
//
// Same operator as qs_policy.cu (SB3 ActorCriticPolicy.forward for MlpPolicy [128,64,64] Tanh;
// reference call sites initial-implementation-v2/rl_train.py:27-53, initial-implementation-v1/rl_train_vecN.py:13-33).
//
// Why: single-pass float16 operands put the value head ~0.7 rms (max ~9) away from the float32 forward because the
// shipped critic has head weights up to 70 (sum |w| = 4000).  Splitting every operand x = hi + lo (two float16, 22
// significant bits) and issuing three MMAs per k-step (hi*hi + hi*lo + lo*hi, float32 accumulation in TMEM) brings the
// error to ~1e-3 on |V| <= 2800 -- the same as torch's own float32 forward -- while the tensor pipe stays far from
// saturated (the kernel is bound by the epilogue's MUFU work, not by MMA issue).
//
// Layout: one persistent CTA per SM, three independent 128-env tiles ("chains", see policy_forward_tc3_kernel).  Shared memory holds
// only the weights (float16 hi and lo, canonical K-major no-swizzle core-matrix layout: offset(row, kchunk) = kchunk*rows*16 +
// row*16 bytes, LBO = rows*16, SBO = 128) and the float32 biases/heads.
// In PRECISE mode weights and biases are pre-multiplied by 2*log2(e), so the accumulator IS the exponent of
// tanh(x) = 1 - 2/(2^acc + 1); four elements share one reciprocal (tanh4_from_exponents): 5 MUFU per 4 tanh, then the hi/lo
// split (LOP3, FADD, 2 F2FP per pair).  Hidden activations never touch shared memory: tcgen05.ld -> registers -> tanh, split
// -> tcgen05.st.
//
// The kernel is launched in single-float16 mode only (QS_POLICY_TENSOR_FAST).  The float32-accurate forward (QS_POLICY_TENSOR)
// runs on the warp-specialised pipeline kernel (qs_rollout_policy.cu), which measured faster than this kernel in PRECISE mode
// (296 vs 308 us per 1M envs, profiles/r02/README.md).
//
// Scheduling, as measured with the clock64 phase trace (QS_TC_TRACE, tools/policy_trace3.py): (1) The MMAs are issued by an elected
// lane under a WARP-UNIFORM branch: from a divergent `if (thread == 0)` each UTCHMMA cost an ELECT/R2UR waterfall (~100 cycles
// per MMA, 8.7k of a tile's 23k cycles).  (2) The observation tile is staged one tile ahead (loaded, normalised, split and stored to
// TMEM while the layer-2 MMAs of the critic run); the tile after that is prefetched into L2.
#include "../../include/quadsim.h"
#include "qs_tc.cuh"
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace qs {
namespace tc {

// (operand layouts, tcgen05/TMEM helpers, tanh and split routines: qs_tc.cuh)
struct Args {
    const float* params;
    const float* obs;
    const float* noise;
    const double* norm;
    float* obs_norm_out;
    float* actions;
    float* actions_clipped;
    float* values;
    float* logp;
    int64_t n;
    float norm_eps, norm_clip;
    float lo[4], hi[4];
};

// Observation row e -> (normalise) -> split float16 -> this lane's 32 TMEM columns at x_addr: the A operand of layer 1.
// Also pulls the row this thread will need one tile later into L2.
template <int OBS, bool PRECISE>
__device__ __forceinline__ void stage_obs_row(const Args& p, int64_t e, bool live, int64_t tile_stride_rows, uint32_t x_addr,
                                              const float* s_mean_hi, const float* s_mean_lo, const float* s_istd) {
    float x[K1];
#pragma unroll
    for (int k = 0; k < K1; ++k) x[k] = 0.f;
    if (live) {
        const float* row = p.obs + e * OBS;
        if (OBS % 4 == 0) {                                     // 80-byte rows: five 16-byte loads
#pragma unroll
            for (int k = 0; k < OBS / 4; ++k) {
                const float4 q = __ldcs(reinterpret_cast<const float4*>(row) + k);
                x[4 * k] = q.x; x[4 * k + 1] = q.y; x[4 * k + 2] = q.z; x[4 * k + 3] = q.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < OBS; ++k) x[k] = __ldcs(row + k);
        }
        const int64_t e_next = e + tile_stride_rows;
        if (e_next < p.n) {
            const char* nr = reinterpret_cast<const char*>(p.obs + e_next * OBS);
            asm volatile("prefetch.global.L2 [%0];" ::"l"(nr));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(nr + OBS * 4 - 4));
        }
        if (p.norm) {
#pragma unroll
            for (int k = 0; k < OBS; ++k) {
                // SB3 subtracts the float64 mean in float64.  Same result to ~2 float32 ulp without FP64 conversions (they run
                // on the XU pipe this kernel is short of): mean = hi + lo in float32; x - hi is exact whenever x is within a
                // factor 2 of the mean (Sterbenz), which is exactly the near-constant-column case that needs the digits.
                const float v = __fmul_rn(__fadd_rn(__fadd_rn(x[k], -s_mean_hi[k]), -s_mean_lo[k]), s_istd[k]);
                x[k] = fminf(fmaxf(v, -p.norm_clip), p.norm_clip);
            }
            if (p.obs_norm_out) {
                float* orow = p.obs_norm_out + e * OBS;
#pragma unroll
                for (int k = 0; k < OBS; ++k) __stcs(orow + k, x[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < OBS; ++k) x[k] = fminf(fmaxf(x[k], -60000.f), 60000.f);   // float16 range
    }
    x[OBS] = 1.0f;                                              // multiplies the bias row of W1
    put32<PRECISE>(x_addr, x);
}

// =====================================================================================================================
// The kernel.  A tile is a serial chain MMA -> epilogue -> MMA ..., so throughput is the number of chains in flight per SM, and
// TMEM (512 columns) is what limits it.  Here a chain needs 160 columns instead of the 232 of whole-layer accumulators:
//     [  0, 64)  R_a: layer-1 accumulator, one 64-output HALF at a time -> in place -> A operand of a partial layer 2;
//                later the layer-3 accumulator
//     [ 64,128)  R_2: layer-2 accumulator (sum of the two partial products) -> in place -> A operand of layer 3
//     [128,160)  observation tile hi | lo
// and column 480 holds the constant (1, 0, ...) chunk for all chains.  Layer 2 is accumulated as the halves of layer 1 finish:
//     L1a -> tanh -> [L2 (+)= H1a.W2[0:64]  and  L1b, issued back to back: MMAs execute in issue order] -> tanh -> L2 += H1b.W2[64:128]
// Three 128-thread groups (one thread per env row, 168 registers available), one tile each: with one warp per scheduler and
// chain the three chains interleave on their own, without turns between the groups.
#ifdef QS_TC_TRACE
__device__ long long g_trace3[3][2][80];
#define QS_TR3() do { if (tr_on && tr_i < 80) g_trace3[g][t >> 5][tr_i++] = clock64(); } while (0)
#else
#define QS_TR3() do { } while (0)
#endif
constexpr int G3 = 3, THREADS3 = G3 * ROWS;
constexpr uint32_t G3_STRIDE = 160, C3_RA = 0, C3_R2 = 64, C3_X = 128, C3_ONE = 480;

// k-steps [0, n_ks) of A (TMEM, chunks of 32 columns: hi at +0, lo at +16) against B k-steps [b_ks0, b_ks0 + n_ks);
// one_col != 0: first the bias k-step (A = constant chunk, B k-step bias_ks).  acc: 0 = overwrite D, 1 = accumulate.
template <bool PRECISE>
__device__ __forceinline__ void issue_part(uint32_t d_col, uint32_t a_col, int n_ks, int b_ks0, uint32_t wb_hi, uint32_t wb_lo, uint32_t b_lbo,
                                           int N, uint32_t acc, uint32_t one_col, int bias_ks) {
    const uint32_t idesc = make_idesc(N);
    if (one_col) {
        umma_ts(d_col, one_col, make_desc(wb_hi + bias_ks * 2 * b_lbo, b_lbo, 128), idesc, acc);
        acc = 1;
        if (PRECISE) umma_ts(d_col, one_col, make_desc(wb_lo + bias_ks * 2 * b_lbo, b_lbo, 128), idesc, 1);
    }
#pragma unroll
    for (int ks = 0; ks < n_ks; ++ks) {
        const uint32_t a_hi = a_col + 32u * (ks >> 1) + 8u * (ks & 1);
        const uint64_t bh = make_desc(wb_hi + (b_ks0 + ks) * 2 * b_lbo, b_lbo, 128);
        umma_ts(d_col, a_hi, bh, idesc, acc);
        acc = 1;
        if (PRECISE) {
            const uint64_t bl = make_desc(wb_lo + (b_ks0 + ks) * 2 * b_lbo, b_lbo, 128);
            umma_ts(d_col, a_hi, bl, idesc, 1);
            umma_ts(d_col, a_hi + 16u, bh, idesc, 1);
        }
    }
}

__device__ __forceinline__ void group_bar3(int g) { asm volatile("bar.sync %0, 128;" ::"r"(g + 1) : "memory"); }

// 64 accumulator columns of this thread's row -> tanh -> in place (hi | lo)
template <bool PRECISE>
__device__ __forceinline__ void epilogue64(uint32_t col) {
    uint32_t v0[32], v1[32];
    float y[32];
    tmem_ld32(col, v0);
    tmem_ld32(col + 32, v1);
    tmem_ld_wait32(v0);
    tanh32<PRECISE>(v0, y);
    put32<PRECISE>(col, y);
    tmem_ld_wait32(v1);
    tanh32<PRECISE>(v1, y);
    put32<PRECISE>(col + 32, y);
}

template <int OBS, bool PRECISE>
__global__ void __launch_bounds__(THREADS3, 1) policy_forward_tc3_kernel(const Args p) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint32_t s_tmem_base;
    __shared__ __align__(8) uint64_t s_bars[G3];
    __shared__ float s_mean[32], s_mean_lo[32], s_istd[32];
    constexpr int OFF_LO = W_SET;
    constexpr int OFF_CONST = PRECISE ? 2 * W_SET : W_SET;
    const int tid = threadIdx.x;
    const int g = tid >> 7, t = tid & 127, warp = tid >> 5;
    const Blob B{OBS};
    float* sC = reinterpret_cast<float*>(smem + OFF_CONST);

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) {
        for (int i = 0; i < G3; ++i) mbar_init(smem_u32(&s_bars[i]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int net = 0; net < 2; ++net) {
        const float sc = PRECISE ? 2.8853900817779268f : 1.0f;
        stage_weights<PRECISE, THREADS3>(p.params + B.w1(net), p.params + B.b1(net), OBS, OBS, K1, N1, sc, smem + OFF_W1 + net * W1_BYTES,
                                         smem + OFF_LO + OFF_W1 + net * W1_BYTES, tid);
        stage_weights<PRECISE, THREADS3>(p.params + B.w2(net), p.params + B.b2(net), N1, N1, N1 + KB, N2, sc, smem + OFF_W2 + net * W2_BYTES,
                                         smem + OFF_LO + OFF_W2 + net * W2_BYTES, tid);
        stage_weights<PRECISE, THREADS3>(p.params + B.w3(net), p.params + B.b3(net), N2, N2, N2 + KB, N3, sc, smem + OFF_W3 + net * W3_BYTES,
                                         smem + OFF_LO + OFF_W3 + net * W3_BYTES, tid);
        for (int i = tid; i < N3 * NACT; i += THREADS3) sC[C_WH + net * N3 * NACT + i] = __ldg(p.params + B.wh(net) + i);
        if (tid < NACT) sC[C_BH + net * NACT + tid] = __ldg(p.params + B.bh(net) + tid);
    }
    if (tid < NACT) sC[C_LS + tid] = __ldg(p.params + B.log_std() + tid);
    if (tid < OBS) {
        double m = 0.0, is = 1.0;
        if (p.norm) {
            m = p.norm[1 + tid];
            is = 1.0 / sqrt(p.norm[1 + OBS + tid] + (double)p.norm_eps);
        }
        s_mean[tid] = (float)m;
        s_mean_lo[tid] = (float)(m - (double)(float)m);
        s_istd[tid] = (float)is;
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // warp-uniform copies for the MMA issuer (first warp of each group)
    const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int g_u = warp_u >> 2;
    const bool issuer_warp = (warp_u & 3) == 0;
    const uint32_t tmem_u = s_tmem_base + (uint32_t)g_u * G3_STRIDE;
    const uint32_t one_u = s_tmem_base + C3_ONE;
    const uint32_t bar_u = smem_u32(&s_bars[0]) + 8u * (uint32_t)g_u;
    const uint32_t lane_bits = (uint32_t)(t & ~31) << 16;
    const uint32_t lane_addr = s_tmem_base + (uint32_t)g * G3_STRIDE + lane_bits;    // this warp's lane quadrant of this group's columns
    const uint32_t bar = smem_u32(&s_bars[g]);
    const uint32_t sbase = smem_u32(smem);
    uint32_t phase = 0;
    constexpr uint32_t B1_LBO = N1 * 16, B2_LBO = N2 * 16;

    if (g == 0) {   // the constant A chunk (1, 0, ..., 0) of the bias k-steps, all 128 lanes, shared by the three chains
        uint32_t one[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) one[j] = 0u;
        one[0] = 0x00003C00u;
        tmem_st16(s_tmem_base + lane_bits + C3_ONE, one);
    }
    const int64_t n_tiles = (p.n + ROWS - 1) / ROWS;
    const int64_t tile_stride = (int64_t)gridDim.x * G3;
    {
        const int64_t tile = (int64_t)blockIdx.x * G3 + g;
        if (tile < n_tiles) {
            const int64_t e = tile * ROWS + t;
            stage_obs_row<OBS, PRECISE>(p, e, e < p.n, tile_stride * ROWS, lane_addr + C3_X, s_mean, s_mean_lo, s_istd);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncthreads();                                                // also publishes group 0's constant chunk to the other groups
    }
    // wait for this group's MMAs: every thread polls the group's mbarrier
    auto mma_wait = [&]() {
        __syncwarp();
        mbar_wait(bar, phase);
        phase ^= 1;
        __syncwarp();
        tc_fence_after();
    };
    auto epilogue_sync = [&]() {
        tmem_st_wait();
        tc_fence_before();
        group_bar3(g);
    };

    for (int64_t tile = (int64_t)blockIdx.x * G3 + g; tile < n_tiles; tile += tile_stride) {
        const int64_t e = tile * ROWS + t;
        const bool live = e < p.n;
#ifdef QS_TC_TRACE
        const bool tr_on = blockIdx.x == 0 && tile == (int64_t)g + 3 * tile_stride && (t == 0 || t == 32);
        int tr_i = 0;
#endif
        QS_TR3();
        float mean[NACT] = {0.f, 0.f, 0.f, 0.f};
        float value = 0.f;
#pragma unroll 1
        for (int net = 0; net < 2; ++net) {
            const uint32_t w1h = sbase + OFF_W1 + net * W1_BYTES, w1l = sbase + OFF_LO + OFF_W1 + net * W1_BYTES;
            const uint32_t w2h = sbase + OFF_W2 + net * W2_BYTES, w2l = sbase + OFF_LO + OFF_W2 + net * W2_BYTES;
            const uint32_t w3h = sbase + OFF_W3 + net * W3_BYTES, w3l = sbase + OFF_LO + OFF_W3 + net * W3_BYTES;
            // ---- layer 1, outputs 0..63: X . W1[:, 0:64] -> R_a
            if (issuer_warp) {
                tc_fence_after();
                if (elect_one()) {
                    issue_part<PRECISE>(tmem_u + C3_RA, tmem_u + C3_X, K1 / 16, 0, w1h, w1l, B1_LBO, 64, 0, 0, 0);
                    umma_commit(bar_u);
                }
            }
            QS_TR3();
            mma_wait();
            QS_TR3();
            epilogue64<PRECISE>(lane_addr + C3_RA);
            QS_TR3();
            epilogue_sync();
            QS_TR3();
            // ---- layer 2 (+)= H1[0:64] . W2[0:64] (with the bias k-step), then layer 1, outputs 64..127 -> R_a
            if (issuer_warp) {
                tc_fence_after();
                if (elect_one()) {
                    issue_part<PRECISE>(tmem_u + C3_R2, tmem_u + C3_RA, 4, 0, w2h, w2l, B2_LBO, N2, 0, one_u, N1 / 16);
                    issue_part<PRECISE>(tmem_u + C3_RA, tmem_u + C3_X, K1 / 16, 0, w1h + 64 * 16, w1l + 64 * 16, B1_LBO, 64, 0, 0, 0);
                    umma_commit(bar_u);
                }
            }
            QS_TR3();
            mma_wait();
            QS_TR3();
            epilogue64<PRECISE>(lane_addr + C3_RA);
            QS_TR3();
            epilogue_sync();
            QS_TR3();
            // ---- layer 2 += H1[64:128] . W2[64:128]
            if (issuer_warp) {
                tc_fence_after();
                if (elect_one()) {
                    issue_part<PRECISE>(tmem_u + C3_R2, tmem_u + C3_RA, 4, 4, w2h, w2l, B2_LBO, N2, 1, 0, 0);
                    umma_commit(bar_u);
                }
            }
            if (net == 1 && tile + tile_stride < n_tiles) {           // next tile's observations, under these MMAs (X is dead)
                const int64_t en = (tile + tile_stride) * ROWS + t;
                stage_obs_row<OBS, PRECISE>(p, en, en < p.n, tile_stride * ROWS, lane_addr + C3_X, s_mean, s_mean_lo, s_istd);
            }
            QS_TR3();
            mma_wait();
            QS_TR3();
            epilogue64<PRECISE>(lane_addr + C3_R2);
            QS_TR3();
            epilogue_sync();
            QS_TR3();
            // ---- layer 3: H2 . W3 -> R_a, then the float32 head
            if (issuer_warp) {
                tc_fence_after();
                if (elect_one()) {
                    issue_part<PRECISE>(tmem_u + C3_RA, tmem_u + C3_R2, N2 / 16, 0, w3h, w3l, B2_LBO, N3, 0, one_u, N2 / 16);
                    umma_commit(bar_u);
                }
            }
            QS_TR3();
            mma_wait();
            QS_TR3();
            float o[NACT];
#pragma unroll
            for (int j = 0; j < NACT; ++j) o[j] = sC[C_BH + net * NACT + j];
            {
                uint32_t v0[32], v1[32];
                float y[32];
                tmem_ld32(lane_addr + C3_RA, v0);
                tmem_ld32(lane_addr + C3_RA + 32, v1);
                tmem_ld_wait32(v0);
                tanh32<PRECISE>(v0, y);
                const float4* wh = reinterpret_cast<const float4*>(sC + C_WH + net * N3 * NACT);
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    const float4 w = wh[k];
                    o[0] = fmaf(y[k], w.x, o[0]); o[1] = fmaf(y[k], w.y, o[1]); o[2] = fmaf(y[k], w.z, o[2]); o[3] = fmaf(y[k], w.w, o[3]);
                }
                tmem_ld_wait32(v1);
                tanh32<PRECISE>(v1, y);
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    const float4 w = wh[32 + k];
                    o[0] = fmaf(y[k], w.x, o[0]); o[1] = fmaf(y[k], w.y, o[1]); o[2] = fmaf(y[k], w.z, o[2]); o[3] = fmaf(y[k], w.w, o[3]);
                }
            }
            if (net == 0) { mean[0] = o[0]; mean[1] = o[1]; mean[2] = o[2]; mean[3] = o[3]; }
            else value = o[0];
            QS_TR3();
            epilogue_sync();
            QS_TR3();      // the next MMAs overwrite R_a, which this thread has just read (and X, if it was re-staged)
        }
        if (live) {
            const float ls[4] = {sC[C_LS], sC[C_LS + 1], sC[C_LS + 2], sC[C_LS + 3]};
            float4 eps = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.noise) eps = __ldcs(reinterpret_cast<const float4*>(p.noise) + e);
            float4 a;
            a.x = fmaf(__expf(ls[0]), eps.x, mean[0]);
            a.y = fmaf(__expf(ls[1]), eps.y, mean[1]);
            a.z = fmaf(__expf(ls[2]), eps.z, mean[2]);
            a.w = fmaf(__expf(ls[3]), eps.w, mean[3]);
            const float HALF_LOG_2PI = 0.9189385332046727f;
            const float lp = -0.5f * (eps.x * eps.x + eps.y * eps.y + eps.z * eps.z + eps.w * eps.w) - (ls[0] + ls[1] + ls[2] + ls[3]) -
                             4.0f * HALF_LOG_2PI;
            __stcs(reinterpret_cast<float4*>(p.actions) + e, a);
            if (p.actions_clipped) {
                float4 c;
                c.x = fminf(fmaxf(a.x, p.lo[0]), p.hi[0]);
                c.y = fminf(fmaxf(a.y, p.lo[1]), p.hi[1]);
                c.z = fminf(fmaxf(a.z, p.lo[2]), p.hi[2]);
                c.w = fminf(fmaxf(a.w, p.lo[3]), p.hi[3]);
                reinterpret_cast<float4*>(p.actions_clipped)[e] = c;
            }
            __stcs(p.values + e, value);
            __stcs(p.logp + e, lp);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s_tmem_base), "r"(TMEM_COLS));
    }
}

}  // namespace tc

#ifdef QS_TC_TRACE
extern "C" int qs_policy_debug_trace3(long long* out_host) {
    return (int)cudaMemcpyFromSymbol(out_host, tc::g_trace3, sizeof(tc::g_trace3));
}
#endif

thread_local char g_policy_tc_error[256] = "";

// single-float16 mode (PRECISE = false) only: see the head of this file
template <int OBS>
static cudaError_t launch_three(const tc::Args& a, int sms, cudaStream_t stream) {
    const int smem = tc::W_SET + tc::C_TOTAL * 4 + 64;
    cudaError_t err = cudaFuncSetAttribute(tc::policy_forward_tc3_kernel<OBS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    const int64_t tiles = (a.n + tc::ROWS - 1) / tc::ROWS;
    const int64_t ctas = (tiles + tc::G3 - 1) / tc::G3;
    const unsigned grid = (unsigned)(ctas < sms ? ctas : sms);
    tc::policy_forward_tc3_kernel<OBS, false><<<grid, tc::THREADS3, smem, stream>>>(a);
    return cudaGetLastError();
}

int launch_policy_tc(const float* params, int obs_dim, const float* obs, const float* noise, int64_t n, const double* norm_stats,
                     float norm_eps, float norm_clip, float* obs_norm_out, float* actions, float* actions_clipped,
                     const float* clip_lo, const float* clip_hi, float* values, float* logp, cudaStream_t stream,
                     const char** err_out) {
    using namespace tc;
    Args a;
    a.params = params; a.obs = obs; a.noise = noise; a.norm = norm_stats; a.obs_norm_out = obs_norm_out;
    a.actions = actions; a.actions_clipped = actions_clipped; a.values = values; a.logp = logp; a.n = n;
    a.norm_eps = norm_eps; a.norm_clip = norm_clip;
    for (int i = 0; i < 4; ++i) { a.lo[i] = clip_lo ? clip_lo[i] : -3.4e38f; a.hi[i] = clip_hi ? clip_hi[i] : 3.4e38f; }
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const cudaError_t err = obs_dim == 20 ? launch_three<20>(a, sms, stream) : launch_three<17>(a, sms, stream);
    if (err != cudaSuccess) {
        snprintf(g_policy_tc_error, sizeof(g_policy_tc_error), "policy_forward_tc3_kernel: %s", cudaGetErrorString(err));
        *err_out = g_policy_tc_error;
        return QS_ECUDA;
    }
    return QS_OK;
}

}  // namespace qs
