// qs_rollout.cu -- ONE kernel per rollout step: VecNormalize normalisation -> MlpPolicy forward on tcgen05 (split-float16,
// float32-class accuracy) -> Gaussian sampling (in-kernel Philox) / log-prob / clipping -> env step (RK4, reward,
// termination, observation, auto-reset) -> VecNormalize batch moments, finalised and merged by the last CTA to finish.
//
// Replaces, for a whole env shard per launch (reference root-relative paths; SB3 = stable_baselines3 2.6.0):
//     OnPolicyAlgorithm.collect_rollouts: policy(obs) -> clip -> env.step      call sites initial-implementation-v2/rl_train.py:27-56,
//                                                                                initial-implementation-v1/rl_train_vecN.py:13-36
//     WaypointQuadEnv.step / reset + DummyVecEnv auto-reset                     initial-implementation-v2/rl_env_scaledObs.py:40-231
//     VecNormalize.step_wait obs_rms.update                                     initial-implementation-v1/rl_train_vecN.py:11
//
// Why one kernel.  The split-float16 policy forward is bound by its epilogues (512 tanh per env: the XU pipe and the issue
// slots), the env step by FMA-pipe work and HBM latency.  Run as separate kernels neither saturates anything (r01: policy
// kernel issue slots 57 %, XU 53 %, tensor 34 %).  Here they share the SM as WARP-SPECIALISED roles of one persistent CTA:
//
//     warps 0-7   epilogue    slot = w >> 2, TMEM lane quadrant = w & 3: tcgen05.ld -> tanh -> hi/lo split -> tcgen05.st, head
//     warps 8-11  env         quadrant = w & 3: observation staging (X operand), sampling, env step, outputs, moments
//     warps 12-13 MMA issue   one per slot: all tcgen05.mma / tcgen05.commit of that slot's tiles
//
// Two SLOTS (256 TMEM columns each: D1[128] | D2[64] | D3[64]) hold two 128-env tiles in flight.  Everything is handed over
// through mbarriers at CHUNK granularity: a layer's MMAs for k-chunk c start as soon as the four epilogue warps of the slot have
// stored chunk c of the previous layer's activations, so only the last chunk's MMAs are exposed; the layer-1 MMAs of the next
// job (a job = one net of one tile) are issued right behind layer 2 of the current one and are long complete when the epilogue
// warps get there.  The X operand (normalised observation tile, hi | lo float16, K-major core-matrix layout) lives in SHARED
// memory (SS form of tcgen05.mma), three buffers, staged two tiles ahead by the env warps; the bias k-steps of layers 2/3 take a
// constant shared-memory A tile, so TMEM holds accumulators/activations only.
//
// Every mbarrier wait is bounded: a protocol error shows up as a sticky status (qs_rollout_status) instead of a hung GPU.
//
// This file is compiled twice (qs_rollout.cu, qs_rollout_policy.cu) with different role configurations -- the fused step wants two
// env warps per scheduler, the policy part alone wants two epilogue warps per (slot, quadrant) -- each in its own namespace QS_RO_NS.
#include "../../include/quadsim.h"
#include "qs_internal.cuh"
#include "qs_tc.cuh"

#include <stdio.h>

#if !defined(QS_RO_NS) || !defined(QS_RO_EPI_SPLIT) || !defined(QS_RO_ENV_SPLIT) || !(defined(QS_RO_BUILD_FUSED) || defined(QS_RO_BUILD_POLICY))
#error "include qs_rollout_impl.cuh from qs_rollout.cu / qs_rollout_policy.cu"
#endif

namespace qs {
namespace QS_RO_NS {
using namespace tc;

// QS_RO_EPI_SPLIT: epilogue warps per (slot, TMEM lane quadrant).  2 = the 32-column chunks of every layer alternate between two
// warps: twice the warps in flight per scheduler (the epilogue is latency-bound per warp: IPC 0.28 measured with one), half the
// epilogue latency of a job.
// QS_RO_ENV_SPLIT: env warps per quadrant.  2 = one env warp per (slot, quadrant): it stages, samples and steps the tiles of its
// slot only, so the env side gets two tile periods per tile (one warp per scheduler was the bottleneck of the fused step).
// With more than 16 warps the launch-time register allowance is below what the env step needs: the roles then re-balance
// registers with setmaxnreg (warpgroups of 4 warps: MMA group gives, env and epilogue groups take).
constexpr int EPI_SPLIT = QS_RO_EPI_SPLIT, ENV_SPLIT = QS_RO_ENV_SPLIT;
// Which of the EPI_SPLIT warps of a (slot, quadrant) takes hidden-layer chunk ch (0-3: layer 1, 4-5: layer 2) and which take the two
// head chunks.  Three warps: (c0, c3, head 0) | (c1, head 1, c4) | (c2, c5) -- 3 / 3 / 2 chunk units per job.
constexpr int HEAD_SPLIT = EPI_SPLIT < 2 ? EPI_SPLIT : 2;
__host__ __device__ constexpr int chunk_owner(int ch) { return EPI_SPLIT == 3 ? (ch < 4 ? ch % 3 : (ch - 3) % 3) : ch % EPI_SPLIT; }
constexpr int EPI_WARPS = 8 * EPI_SPLIT, ENV_WARPS = 4 * ENV_SPLIT, MMA_WARPS = 2;
// A/B switch (QS_RO_ENV_FIRST): which role gets the low warp ids -- the schedulers favour older (lower) warps when several are
// ready, and the env warps' few MUFU ops queue behind the epilogue warps' thousands
#ifndef QS_RO_ENV_FIRST
#define QS_RO_ENV_FIRST 0
#endif
#ifndef QS_RO_LDBUF
#define QS_RO_LDBUF 1
#endif
// QS_RO_LD_SPLIT: the epilogue loads a 32-column chunk as two 16-column halves and converts the first while the second is in
// flight (tcgen05.ld latency off the warp's critical path); needs the k-step-local activation layout (see issue_chunk)
#ifndef QS_RO_LD_SPLIT
#define QS_RO_LD_SPLIT 0
#endif
// QS_RO_ST16: the epilogue stores a converted chunk with two 16-column tcgen05.st from ONE address register instead of eight 4-column
// ones (each needs its address in a uniform register: 9 R2UR + 12 register moves per chunk in the SASS).  Policy build (80 registers):
// 275.1 -> 266.5 us per 1M-env launch; the fused build's epilogue warps (72 / 88 registers) get slower with it (378 -> 392 us).
#ifndef QS_RO_ST16
#ifdef QS_RO_BUILD_POLICY
#define QS_RO_ST16 1
#else
#define QS_RO_ST16 0
#endif
#endif
constexpr int W_EPI0 = QS_RO_ENV_FIRST ? ENV_WARPS : 0, W_ENV0 = QS_RO_ENV_FIRST ? 0 : EPI_WARPS, W_MMA0 = EPI_WARPS + ENV_WARPS;
// the block is padded to whole groups of 4 warps: registers are allocated per 4 warps anyway (a 448 x 144 launch is refused)
constexpr int RO_WARPS = ((EPI_WARPS + ENV_WARPS + MMA_WARPS + 3) / 4) * 4;
constexpr int RO_THREADS = RO_WARPS * 32;
constexpr int REGS_LAUNCH = (65536 / RO_THREADS) / 8 * 8;
// setmaxnreg targets (multiples of 8), used when the launch allowance is below 128: what is left after the MMA group dropped to 40
#ifdef QS_RO_BUILD_FUSED
constexpr bool REBALANCE = REGS_LAUNCH < 128;
#else
constexpr bool REBALANCE = false;      // the policy part alone fits the launch allowance
#endif
constexpr int REGS_MMA = 40;
constexpr int REGS_ENV = EPI_SPLIT == 1 ? 128 : 152;
constexpr int REGS_EPI = EPI_SPLIT == 1 ? 88 : 72;
// setmaxnreg moves registers inside the CTA's own launch-time allocation only (the pool is per CTA: an increase beyond what the
// other warpgroups have released blocks forever -- measured the hard way)
static_assert(!REBALANCE || (EPI_WARPS * REGS_EPI + ENV_WARPS * REGS_ENV + 4 * REGS_MMA) * 32 <= RO_THREADS * REGS_LAUNCH, "register pool of the CTA");
static_assert(!REBALANCE || (EPI_WARPS % 4 == 0 && ENV_WARPS % 4 == 0), "setmaxnreg works on whole warpgroups");
// X operand buffers: with one env warp per (slot, quadrant) the slot's buffer is free again (its critic's layer 1 long complete) when
// that warp stages the slot's next tile, so one buffer per slot suffices; a single env warp per quadrant stages two tiles ahead
constexpr int XBUFS = ENV_SPLIT == 2 ? 2 : 3;

constexpr uint32_t SLOT_COLS = 256, C_D1 = 0, C_D2 = 128, C_D3 = 192;

// ---- the policy image: what every CTA copies verbatim into the front of its shared memory ------------------------------
constexpr int IMG_WHI = 0, IMG_WLO = W_SET, IMG_CONST = 2 * W_SET;
constexpr int IMG_BYTES = IMG_CONST + ((C_TOTAL * 4 + 127) / 128) * 128;  // 131072 + 4224
// ---- the rest of the shared-memory map ----------------------------------------------------------------------------------
constexpr int X_HALF = (K1 / 8) * ROWS * 16;                               // 8192: one precision part of an X tile
constexpr int X_BYTES = 2 * X_HALF;
constexpr int ONE_BYTES = 2 * ROWS * 16;                                   // 128 rows x 16 K float16
constexpr int X_LBO = ROWS * 16;                                           // K-direction stride between core matrices
constexpr int SM_ONE = IMG_BYTES;
constexpr int SM_X = SM_ONE + ONE_BYTES;
constexpr int SM_OUT_MEAN = SM_X + XBUFS * X_BYTES;                        // float4[2][HEAD_SPLIT][128] partial head sums
constexpr int SM_OUT_VAL = SM_OUT_MEAN + 2 * HEAD_SPLIT * ROWS * 16;       // float[2][HEAD_SPLIT][128]
constexpr int SM_TILE = SM_OUT_VAL + 2 * HEAD_SPLIT * ROWS * 4;                         // float[ENV_WARPS][32 * 21]
constexpr int SM_MOM = SM_TILE + ENV_WARPS * 32 * 21 * 4;                  // double[ENV_WARPS][2 * 20]
constexpr int SM_NORM = SM_MOM + ENV_WARPS * 40 * 8;                       // float[3][32]
constexpr int SM_BARS = SM_NORM + 3 * 32 * 4;
enum : int { B_XFULL = 0 /* [3] */, B_XFREE = 3 /* [3] */, B_D1 = 6, B_D2 = 8, B_D3 = 10, B_H1 = 12, B_H2 = 20, B_D3FREE = 24, B_OUTF = 26, B_OUTE = 34, N_BARS = 42 };
constexpr int SM_MISC = SM_BARS + N_BARS * 8;                              // tmem base, last-CTA flag
constexpr int SM_TOTAL = SM_MISC + 16;
static_assert(SM_TOTAL <= 232448, "shared memory budget of one CTA on B200");
static_assert(SM_X % 128 == 0 && SM_ONE % 128 == 0, "operand tiles are 128-byte aligned");

__device__ int g_ro_status;          // sticky: != 0 after a bounded wait expired (role * 100 + barrier index + 1)

// Development aid (-DQS_RO_TRACE=1, tools/rollout_trace.py): lane 0 of every warp of CTA 0 logs (event code, clock) pairs, so the
// hand-over latencies between the roles can be read off a real run.  Compiled out of the product build.
#ifdef QS_RO_TRACE
constexpr int TRACE_LEN = 2048;
__device__ uint2 g_ro_trace[32][TRACE_LEN];
#define RO_TRACE_INIT() uint2* tr_buf = g_ro_trace[threadIdx.x >> 5]; int tr_n = 0; const bool tr_on = blockIdx.x == 0 && (threadIdx.x & 31) == 0
#define RO_TRACE(code) do { if (tr_on && tr_n < TRACE_LEN - 1) tr_buf[tr_n++] = make_uint2((uint32_t)(code), (uint32_t)clock64()); } while (0)
#define RO_TRACE_END() do { if (tr_on) tr_buf[TRACE_LEN - 1] = make_uint2((uint32_t)tr_n, 0u); } while (0)
#else
#define RO_TRACE_INIT() do { } while (0)
#define RO_TRACE(code) do { } while (0)
#define RO_TRACE_END() do { } while (0)
#endif

struct RoParams {
    // policy
    const unsigned char* image;      // prepared operand image (IMG_BYTES), or null -> stage from `params`
    const float* params;             // raw float32 blob (qs_policy_forward layout)
    const float* obs;                // [n, OBS]
    const double* norm;              // VecNormalize stats or null
    float norm_eps, norm_clip;
    int sample_mode;                 // QS_SAMPLE_*
    const float* noise;              // [n, 4]
    uint64_t noise_seed;
    unsigned long long* noise_step;  // device counter word (QS_SAMPLE_PHILOX)
    float lo[4], hi[4];
    float* obs_norm_out;
    float* actions;                  // unclipped
    float* actions_clipped;          // or null
    float* values;
    float* logp;
    int64_t n;
    // env step (FUSED)
    StepParams<float> sp;
    double* mom_out;                 // (n, mean, M2) triplet or null
    double* mom_merge;               // running statistics to merge into, or null
    unsigned int* ticket;            // last-CTA election counter (handle-owned, zero between launches)
};

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded parity wait (all lanes poll).  false = gave up: the caller leaves its role, the status word says where.
// A plain try_wait loop returns every ~30 cycles; with ten warps of an SM waiting most of the time the polling alone was 40 % of
// all issued instructions (ncu, profiles/r02) and starved the warps that had work.  So: the suspend-time hint of try_wait (the
// thread sleeps in the barrier unit until the phase completes, the hint expires or -- as measured -- another barrier of the CTA is hit).
// No nanosleep between polls: `nanosleep.u32` has a coarse granularity here (a 20 ns and a 500 ns request cost the same, and made
// every hand-over slower: 294 -> 336 us for the policy part).
#ifndef QS_RO_WAIT_HINT_NS
#define QS_RO_WAIT_HINT_NS 20000
#endif
#ifndef QS_RO_BACKOFF_NS
#define QS_RO_BACKOFF_NS 0
#endif
__device__ __forceinline__ uint32_t mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
#if QS_RO_WAIT_HINT_NS > 0
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"((uint32_t)QS_RO_WAIT_HINT_NS)
        : "memory");
#else
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
#endif
    return ok;
}
// non-blocking probe
__device__ __forceinline__ uint32_t mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}
// QS_RO_TIGHT_WAIT (r02): the whole bounded wait is ONE asm block -- try_wait (hinted), branch, counter -- 5 SASS instructions per
// wake-up instead of the ~16 the C loop compiled to.  A parked warp is woken by every barrier event of the CTA (measured: ~7.7M
// wake-ups per 1M-env launch), and with the epilogue warps busy back to back those wake-ups competed for issue slots that were
// 72 % taken (ncu): the loop's length is a cost, not a detail.  The bound stays: 2^22 wake-ups (seconds), then the sticky status.
#ifndef QS_RO_TIGHT_WAIT
#define QS_RO_TIGHT_WAIT 1
#endif
__device__ __forceinline__ bool mbar_wait_slow(uint32_t bar, uint32_t parity, int code) {
#if QS_RO_TIGHT_WAIT
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        ".reg .u32 n;\n\t"
        "mov.u32 n, 0;\n\t"
        "QS_WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "@p bra QS_WAIT_DONE;\n\t"
        "add.u32 n, n, 1;\n\t"
        "setp.lt.u32 q, n, 4194304;\n\t"
        "@q bra QS_WAIT_LOOP;\n\t"
        "QS_WAIT_DONE:\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"((uint32_t)(QS_RO_WAIT_HINT_NS > 0 ? QS_RO_WAIT_HINT_NS : 1000))
        : "memory");
    if (ok) return true;
#else
    for (uint32_t it = 0; it < (1u << 17); ++it) {                 // x (up to) 20 us per try: seconds, not minutes
#if QS_RO_BACKOFF_NS > 0
        __nanosleep(QS_RO_BACKOFF_NS);
#endif
        if (mbar_try(bar, parity)) return true;
        if ((it & 0xFF) == 0xFF && *reinterpret_cast<volatile int*>(&g_ro_status) != 0) break;   // somebody else already gave up
    }
#endif
    atomicCAS(&g_ro_status, 0, code);
    return false;
}
__device__ __forceinline__ bool mbar_wait_bounded(uint32_t bar, uint32_t parity, int code) {
    if (mbar_try(bar, parity)) return true;
    return mbar_wait_slow(bar, parity, code);
}
// The same for a wait that is NOT on the critical path (the env warps' wait for a tile's outputs, which they consume a whole tile
// period late): a hinted try_wait is woken by EVERY barrier event of the CTA -- measured 83 wake-ups per output wait, 2.7 M per
// 1M-env launch, ~8 % of all issued instructions, taken from the epilogue warps' issue slots -- so this one sleeps on the timer
// between probes instead (nanosleep is coarse, ~0.5-1 us: far below the tile period of ~5 us).
#ifndef QS_RO_LAZY_WAIT_NS
#define QS_RO_LAZY_WAIT_NS 600
#endif
__device__ __forceinline__ bool mbar_wait_lazy(uint32_t bar, uint32_t parity, int code) {
#if QS_RO_LAZY_WAIT_NS > 0
    if (mbar_test(bar, parity)) return true;
    for (uint32_t it = 0; it < (1u << 22); ++it) {                 // x ~1 us: seconds, then the sticky status
        __nanosleep(QS_RO_LAZY_WAIT_NS);
        if (mbar_test(bar, parity)) return true;
    }
    atomicCAS(&g_ro_status, 0, code);
    return false;
#else
    return mbar_wait_bounded(bar, parity, code);
#endif
}
// D[tmem] (+)= A[smem] . B[smem]^T
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// (a, b) -> packed float16 hi (round to nearest) and packed lo = exact remainders: F2FP + 2 FHFMA + F2FP per pair (the
// LOP3 / FADD / 2 x F2FP sequence of qs_tc.cuh::split_h2 costs 6)
__device__ __forceinline__ void split_h2_rn(float a, float b, uint32_t& hi, uint32_t& lo) {
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
#ifdef QS_X_NOSPLIT                          // timing experiment only (wrong numerics): what the lo half costs
    lo = hi ^ 0x3C003C00u;
    return;
#endif
#ifdef QS_X_TRUNCSPLIT                       // A/B: hi by truncation (LOP3 on the ALU pipe), lo = exact remainder by FADD (r01's split)
    split_h2(a, b, hi, lo);
    return;
#endif
    float la, lb;
    asm("{\n\t"
        ".reg .f16 l, h, m;\n\t"
        "mov.b32 {l, h}, %2;\n\t"
        "mov.b16 m, 0xBC00;\n\t"                       // -1.0: lo = x - hi as one mixed-precision FMA
        "fma.rn.f32.f16 %0, l, m, %3;\n\t"
        "fma.rn.f32.f16 %1, h, m, %4;\n\t"
        "}\n"
        : "=f"(la), "=f"(lb)
        : "r"(hi), "f"(a), "f"(b));
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(lb), "f"(la));
}
// y[32] -> packed hi (16 columns at taddr) | lo (16 columns at taddr + 16), in place over the accumulator chunk
__device__ __forceinline__ void put32_rn(uint32_t taddr, const float* y) {
    uint32_t h[16], l[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) split_h2_rn(y[2 * j], y[2 * j + 1], h[j], l[j]);
    tmem_st16(taddr, h);
    tmem_st16(taddr + 16, l);
}

struct Ctx {
    uint32_t sbase;       // shared-memory window address of the dynamic buffer
    uint32_t tmem;        // TMEM base
    int cnt;              // 128-env tiles of this CTA: tile(i) = blockIdx.x + i * gridDim.x
    __device__ __forceinline__ uint32_t bar(int idx) const { return sbase + SM_BARS + 8u * (uint32_t)idx; }
};

// ---------------------------------------------------------------------------------------------------------------------
// MMA issuer of one slot.  All lanes wait on the mbarriers (warp-uniform control flow), one elected lane issues.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void issue_l1(const Ctx& c, uint32_t d1, int xb, int net) {
    const uint32_t idesc = make_idesc(N1);
    const uint32_t xa = c.sbase + SM_X + xb * X_BYTES;
    const uint32_t wh = c.sbase + IMG_WHI + OFF_W1 + net * W1_BYTES, wl = c.sbase + IMG_WLO + OFF_W1 + net * W1_BYTES;
    constexpr uint32_t B_LBO = N1 * 16;
#pragma unroll
    for (int ks = 0; ks < K1 / 16; ++ks) {
        const uint64_t ah = make_desc(xa + ks * 2 * X_LBO, X_LBO, 128), al = make_desc(xa + X_HALF + ks * 2 * X_LBO, X_LBO, 128);
        const uint64_t bh = make_desc(wh + ks * 2 * B_LBO, B_LBO, 128), bl = make_desc(wl + ks * 2 * B_LBO, B_LBO, 128);
        umma_ss(d1, ah, bh, idesc, ks ? 1u : 0u);
        umma_ss(d1, ah, bl, idesc, 1);
        umma_ss(d1, al, bh, idesc, 1);
    }
}
// bias k-step: D = ONE . Bbias (hi, lo), overwriting D
__device__ __forceinline__ void issue_bias(const Ctx& c, uint32_t d, uint32_t wh, uint32_t wl, int bias_ks) {
    constexpr uint32_t B_LBO = N2 * 16;
    const uint32_t idesc = make_idesc(N2);
    const uint64_t one = make_desc(c.sbase + SM_ONE, X_LBO, 128);
    umma_ss(d, one, make_desc(wh + bias_ks * 2 * B_LBO, B_LBO, 128), idesc, 0);
    umma_ss(d, one, make_desc(wl + bias_ks * 2 * B_LBO, B_LBO, 128), idesc, 1);
}
// the two k-steps of activation chunk `ch` (32 columns at a_col: hi | lo) against the matching weight k-steps
__device__ __forceinline__ void issue_chunk(uint32_t d, uint32_t a_col, int ch, uint32_t wh, uint32_t wl) {
    constexpr uint32_t B_LBO = N2 * 16;
    const uint32_t idesc = make_idesc(N2);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int ks = 2 * ch + j;
        // activation layout inside a 32-column chunk: QS_RO_LD_SPLIT = 0: [hi k-step 0 | hi k-step 1 | lo 0 | lo 1] (8 columns each);
        // = 1: [hi 0 | lo 0 | hi 1 | lo 1], i.e. each k-step's 16 activations stay inside their own 16 columns
        const uint32_t a_hi = a_col + 32u * ch + (QS_RO_LD_SPLIT ? 16u : 8u) * j;
        const uint64_t bh = make_desc(wh + ks * 2 * B_LBO, B_LBO, 128), bl = make_desc(wl + ks * 2 * B_LBO, B_LBO, 128);
        umma_ts(d, a_hi, bh, idesc, 1);
        umma_ts(d, a_hi, bl, idesc, 1);
        umma_ts(d, a_hi + (QS_RO_LD_SPLIT ? 8u : 16u), bh, idesc, 1);
    }
}

__device__ __forceinline__ void role_mma(const Ctx& c, int slot) {
    const uint32_t d1 = c.tmem + slot * SLOT_COLS + C_D1, d2 = c.tmem + slot * SLOT_COLS + C_D2, d3 = c.tmem + slot * SLOT_COLS + C_D3;
    const int role = 300 + slot * 50;
    uint32_t job = 0;
    bool l1_issued = false;
    RO_TRACE_INIT();
    for (int i = slot; i < c.cnt; i += 2) {
        const int xb = i % XBUFS;
#pragma unroll 1
        for (int net = 0; net < 2; ++net, ++job) {
            const uint32_t par = job & 1u;
            const uint32_t w2h = c.sbase + IMG_WHI + OFF_W2 + net * W2_BYTES, w2l = c.sbase + IMG_WLO + OFF_W2 + net * W2_BYTES;
            const uint32_t w3h = c.sbase + IMG_WHI + OFF_W3 + net * W3_BYTES, w3l = c.sbase + IMG_WLO + OFF_W3 + net * W3_BYTES;
            if (!l1_issued) {                                   // the slot's first job, or the X tile was not ready when layer 2 went out
                if (net == 0 && !mbar_wait_bounded(c.bar(B_XFULL + xb), (uint32_t)(i / XBUFS) & 1u, role + B_XFULL + 1)) return;
                tc_fence_after();
                if (elect_one()) {
                    issue_l1(c, d1, xb, net);
                    umma_commit(c.bar(B_D1 + slot));
                    if (net == 1) umma_commit(c.bar(B_XFREE + xb));
                }
                __syncwarp();
                RO_TRACE(0x200000u | job);
            }
            l1_issued = false;
            // ---- layer 2: bias k-step, then the chunks of H1 as the epilogue warps deliver them
            if (elect_one()) issue_bias(c, d2, w2h, w2l, N1 / 16);
            __syncwarp();
#pragma unroll 1
            for (int ch = 0; ch < 4; ++ch) {
                if (!mbar_wait_bounded(c.bar(B_H1 + slot * 4 + ch), par, role + B_H1 + 1)) return;
                RO_TRACE(0x210000u | (ch << 12) | job);
                tc_fence_after();
                if (elect_one()) {
                    issue_chunk(d2, d1, ch, w2h, w2l);
                    if (ch == 3) umma_commit(c.bar(B_D2 + slot));
                }
                __syncwarp();
            }
            RO_TRACE(0x220000u | job);
            // ---- layer 1 of the NEXT job right behind (MMAs execute in issue order: D1 is free once layer 2 has read it) -- unless it
            // needs an X tile the env warps have not staged yet: then layer 3 of this job goes first (no head-of-line blocking)
            int nxb = xb, nnet = 1, ni = i;
            bool have_next = true;
            if (net == 1) { ni = i + 2; nnet = 0; nxb = ni % XBUFS; have_next = ni < c.cnt; }
            bool l1_now = have_next && (net == 0 || mbar_test(c.bar(B_XFULL + nxb), (uint32_t)(ni / XBUFS) & 1u));
            l1_now = __shfl_sync(0xffffffffu, l1_now ? 1 : 0, 0) != 0;
            if (l1_now) {
                tc_fence_after();
                if (elect_one()) {
                    issue_l1(c, d1, nxb, nnet);
                    umma_commit(c.bar(B_D1 + slot));
                    if (nnet == 1) umma_commit(c.bar(B_XFREE + nxb));          // the critic is the X tile's last reader
                }
                __syncwarp();
                l1_issued = true;
                RO_TRACE(0x230000u | job);
            }
            // ---- layer 3 (D3 is free once the epilogue warps have loaded the previous job's layer-3 result)
            if (!mbar_wait_bounded(c.bar(B_D3FREE + slot), par ^ 1u, role + B_D3FREE + 1)) return;
            RO_TRACE(0x240000u | job);
            tc_fence_after();
            if (elect_one()) issue_bias(c, d3, w3h, w3l, N2 / 16);
            __syncwarp();
#pragma unroll 1
            for (int ch = 0; ch < 2; ++ch) {
                if (!mbar_wait_bounded(c.bar(B_H2 + slot * 2 + ch), par, role + B_H2 + 1)) return;
                RO_TRACE(0x250000u | (ch << 12) | job);
                tc_fence_after();
                if (elect_one()) {
                    issue_chunk(d3, d2, ch, w3h, w3l);
                    if (ch == 1) umma_commit(c.bar(B_D3 + slot));
                }
                __syncwarp();
            }
            RO_TRACE(0x260000u | job);
        }
    }
    RO_TRACE_END();
}
// the first job of a slot issues the critic's L1 from inside the loop above (net == 0 -> next job is net 1 of the same tile), so
// the X buffer of that tile is released there too.

// ---------------------------------------------------------------------------------------------------------------------
// Epilogue warp (slot, quadrant): 32 env rows = its TMEM lanes.
// ---------------------------------------------------------------------------------------------------------------------
// The hot loops are ROLLED on purpose: B200's instruction caches are small (L0 ~6 KB per scheduler, L1.5 32 KB per SM) and four
// different instruction streams share them here.  With the epilogues unrolled per chunk the kernel's hot code was ~100 KB and
// `no_inst` (instruction fetch) was the top stall of every role (ncu, profiles/r02); one ~5 KB chunk routine serves all
// six hidden-layer chunks, another the two head chunks.
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
}
// One 32-column accumulator chunk of this lane's row at `col`: tcgen05.ld -> tanh -> hi | lo split, stored in place over the chunk
// (hi halves in columns [0,16), lo halves in [16,32)).  Eight activations at a time keep the live registers near 64.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t* v) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]),
                   "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :
                 : "memory");
}
// eight activations of this lane's row: tanh -> hi | lo packed halves stored at hi_col / lo_col (4 columns each)
__device__ __forceinline__ void tanh_split8(const uint32_t* v, uint32_t hi_col, uint32_t lo_col) {
    float y[8];
    tanh8_from_exponents(v, y);
    uint32_t h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) split_h2_rn(y[2 * j], y[2 * j + 1], h[j], l[j]);
    tmem_st4(hi_col, h);
    tmem_st4(lo_col, l);
}
__device__ __forceinline__ void chunk_tanh_split(uint32_t col) {
    uint32_t v[32];
#if QS_RO_LD_SPLIT
    tmem_ld16(col, v);
    tmem_ld_wait16(v);
    tmem_ld16(col + 16u, v + 16);                     // in flight while the first 16 activations are converted (they stay inside columns [0, 16))
    tanh_split8(v, col, col + 8u);
    tanh_split8(v + 8, col + 4u, col + 12u);
    tmem_ld_wait16(v + 16);
    tanh_split8(v + 16, col + 16u, col + 24u);
    tanh_split8(v + 24, col + 20u, col + 28u);
#else
    tmem_ld32(col, v);
    tmem_ld_wait32(v);
#if QS_RO_ST16                                   // A/B: two 16-column stores per chunk (one address, no per-store R2UR) instead of eight 4-column ones
    uint32_t h[16], l[16];
#pragma unroll
    for (int sb = 0; sb < 4; ++sb) {
        float y[8];
        tanh8_from_exponents(v + 8 * sb, y);
#pragma unroll
        for (int j = 0; j < 4; ++j) split_h2_rn(y[2 * j], y[2 * j + 1], h[4 * sb + j], l[4 * sb + j]);
    }
    asm volatile(
        "{\n\t"
        ".reg .b32 a2;\n\t"
        "add.u32 a2, %0, 16;\n\t"
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n\t"
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [a2], {%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n\t"
        "}\n" ::"r"(col),
        "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]), "r"(h[4]), "r"(h[5]), "r"(h[6]), "r"(h[7]), "r"(h[8]), "r"(h[9]), "r"(h[10]), "r"(h[11]), "r"(h[12]),
        "r"(h[13]), "r"(h[14]), "r"(h[15]), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]), "r"(l[4]), "r"(l[5]), "r"(l[6]), "r"(l[7]), "r"(l[8]), "r"(l[9]),
        "r"(l[10]), "r"(l[11]), "r"(l[12]), "r"(l[13]), "r"(l[14]), "r"(l[15])
        : "memory");
#else
#pragma unroll
    for (int sb = 0; sb < 4; ++sb) tanh_split8(v + 8 * sb, col + 4u * sb, col + 16u + 4u * sb);
#endif
#endif
}

// Order of a warp's work (QS_RO_DEFER_HEAD, r02): the head of job j-1 runs BETWEEN the layer-1 and the layer-2 epilogue of job j,
//     E1(j) -> head(j-1) -> E2(j) -> E1(j+1) -> head(j) -> E2(j+1) -> ...
// instead of E1(j) -> E2(j) -> head(j).  In the straight order the warp idles twice per job -- after E1 until the last two chunks'
// MMAs have produced D2 (800-1,800 cycles) and after E2 until D3 (700-1,150; phase trace, profiles/r02) -- 40 % of a job.  Deferred,
// every wait has a whole phase of other work in front of it: D3(j-1) has had E1(j) to complete, D2(j) completes under head(j-1), and
// D1(j+1) (issued behind layer 2 of job j) under head(j-1) + E2(j).  Nothing else changes: D3 is not overwritten before layer 3 of
// job j, which the MMA warp issues after E2(j) and after D3FREE, i.e. after head(j-1).  The env warps consume a tile's outputs one
// iteration later to match (LAG in role_env).
#ifndef QS_RO_DEFER_HEAD
#define QS_RO_DEFER_HEAD 1
#endif
// QS_RO_HEAD_SCALAR_VF: the critic's head has one output -- a scalar weight and one FFMA per activation instead of the actor's float4 and
// four.  Policy build: 280.1 -> 276.2 us; the fused build (one epilogue warp per (slot, quadrant), larger code) gets slower with the
// second head body (374.5 -> 389.9 us): off there.
#ifndef QS_RO_HEAD_SCALAR_VF
#ifdef QS_RO_BUILD_POLICY
#define QS_RO_HEAD_SCALAR_VF 1
#else
#define QS_RO_HEAD_SCALAR_VF 0
#endif
#endif
__device__ __forceinline__ void role_epilogue(const Ctx& c, int slot, int half, int quad, int lane, const float* sC, float4* s_mean, float* s_val) {
    const uint32_t tm = c.tmem + slot * SLOT_COLS + ((uint32_t)(quad * 32) << 16);
    const int role = 100 + slot * 50;
    const int row = quad * 32 + lane;
    const uint32_t njobs = c.cnt > slot ? 2u * (uint32_t)((c.cnt - slot + 1) / 2) : 0u;    // two jobs (actor, critic) per tile of this slot
    float mean[NACT] = {0.f, 0.f, 0.f, 0.f};
    RO_TRACE_INIT();
    // iteration `job` does E1(job), head(job - DEFER), E2(job); one extra iteration drains the last head
#pragma unroll 1
    for (uint32_t job = 0; job < njobs + QS_RO_DEFER_HEAD; ++job) {
        const uint32_t par = job & 1u;
        const bool live = job < njobs;
        // chunks 0-3: layer-1 accumulator D1 -> H1; chunks 4-5: layer-2 accumulator D2 -> H2 (D2 follows D1 in the slot's columns);
        // this warp takes every EPI_SPLIT-th chunk.  Each: tcgen05.ld -> tanh -> hi | lo in place -> signal the MMA warp.
#pragma unroll 1
        for (int stage = 0; stage < 3; ++stage) {
            if (stage == (QS_RO_DEFER_HEAD ? 1 : 2)) {
                // ---- head of job hj: layer-3 accumulator D3 -> tanh -> partial sums against the float32 head weights
                if (QS_RO_DEFER_HEAD ? job == 0 : !live) continue;
                if (half >= HEAD_SPLIT) continue;                            // (with three warps the third has no head chunk)
                const uint32_t hj = job - QS_RO_DEFER_HEAD, hpar = hj & 1u;
                const int net = (int)(hj & 1u);
                const uint32_t k = hj >> 1;                                  // this slot's tile counter
                if (!mbar_wait_bounded(c.bar(B_D3 + slot), hpar, role + B_D3 + 1)) return;
                RO_TRACE(0x130000u | hj);
                tc_fence_after();
                float o[NACT];                                               // partial head sums of this warp's chunks (+ bias in half 0)
#pragma unroll
                for (int j = 0; j < NACT; ++j) o[j] = half == 0 ? sC[C_BH + net * NACT + j] : 0.f;
#pragma unroll 1
                for (int ch = half; ch < 2; ch += HEAD_SPLIT) {
                    uint32_t v[32];
                    tmem_ld32(tm + C_D3 + 32u * (uint32_t)ch, v);
                    tmem_ld_wait32(v);
                    if (ch + HEAD_SPLIT >= 2) {                               // this warp's last read of D3: layer 3 of the next job may overwrite it
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(c.bar(B_D3FREE + slot));
                    }
                    const float4* wh = reinterpret_cast<const float4*>(sC + C_WH + net * N3 * NACT) + 32 * ch;
#pragma unroll
                    for (int sb = 0; sb < 4; ++sb) {
                        float y[8];
                        tanh8_from_exponents(v + 8 * sb, y);
#if QS_RO_HEAD_SCALAR_VF
                        if (net == 1) {                                      // the critic's head has ONE output: a scalar weight and one FFMA per activation
                            const float* w1 = reinterpret_cast<const float*>(wh + 8 * sb);
#pragma unroll
                            for (int q = 0; q < 8; ++q) o[0] = fmaf(y[q], w1[4 * q], o[0]);
                        } else
#endif
                        {
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                                const float4 w = wh[8 * sb + q];
                                o[0] = fmaf(y[q], w.x, o[0]); o[1] = fmaf(y[q], w.y, o[1]); o[2] = fmaf(y[q], w.z, o[2]); o[3] = fmaf(y[q], w.w, o[3]);
                            }
                        }
                    }
                }
                RO_TRACE(0x140000u | hj);
                if (net == 0) {
#pragma unroll
                    for (int j = 0; j < NACT; ++j) mean[j] = o[j];
                } else {
                    if (!mbar_wait_bounded(c.bar(B_OUTE + slot * 4 + quad), (k & 1u) ^ 1u, role + B_OUTE + 1)) return;
                    s_mean[(slot * HEAD_SPLIT + half) * ROWS + row] = make_float4(mean[0], mean[1], mean[2], mean[3]);
                    s_val[(slot * HEAD_SPLIT + half) * ROWS + row] = o[0];
                    __syncwarp();
                    if (lane == 0) mbar_arrive(c.bar(B_OUTF + slot * 4 + quad));
                }
            } else {
                // ---- E1 (first stage) or E2 of job `job`
                if (!live) continue;
                const bool first = stage == 0;
                if (EPI_SPLIT == 3 && !first && half == 0) continue;         // owns no layer-2 chunk
                if (!mbar_wait_bounded(c.bar((first ? B_D1 : B_D2) + slot), par, role + (first ? B_D1 : B_D2) + 1)) return;
                tc_fence_after();
#pragma unroll 1
                for (int ch = (first ? 0 : 4); ch < (first ? 4 : 6); ++ch) {
                    if (chunk_owner(ch) != half) continue;
                    RO_TRACE(0x100000u | (ch << 12) | job);
                    chunk_tanh_split(tm + 32u * (uint32_t)ch);
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(c.bar(first ? B_H1 + slot * 4 + ch : B_H2 + slot * 2 + (ch - 4)));
                    RO_TRACE(0x110000u | (ch << 12) | job);
                }
            }
        }
    }
    RO_TRACE_END();
}

// ---------------------------------------------------------------------------------------------------------------------
// Env warp (quadrant): stages the X operand two tiles ahead, then per tile: policy outputs -> sample -> (env step) -> stores.
// ---------------------------------------------------------------------------------------------------------------------
// standard normal noise of (seed, global env id, step): Philox4x32-10 -> two Box-Muller pairs
__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint64_t gid, unsigned long long step) {
    uint32_t w[4];
    philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)step, (uint32_t)(step >> 32), (uint32_t)seed ^ 0x85A308D3u,
                  (uint32_t)(seed >> 32) ^ 0x243F6A88u, w);
    float z[4];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float u1 = ((float)(w[2 * j] >> 9) + 0.5f) * 1.1920928955078125e-07f;             // (0, 1), 23 bits
        const float th = (float)(w[2 * j + 1] >> 8) * 3.7450702829239286e-07f;                  // [0, 2 pi): 2 pi * 2^-24
        const float r = sqrtf(-1.3862943611198906f * __log2f(u1));                              // sqrt(-2 ln u1)
        float s, co;
        __sincosf(th, &s, &co);
        z[2 * j] = r * co;
        z[2 * j + 1] = r * s;
    }
    return make_float4(z[0], z[1], z[2], z[3]);
}

template <int OBS>
__device__ __forceinline__ bool stage_x(const Ctx& c, const RoParams& p, int i, int quad, int lane, unsigned char* smem, const float* s_norm) {
    const int xb = i % XBUFS;
    if (!mbar_wait_bounded(c.bar(B_XFREE + xb), ((uint32_t)(i / XBUFS) & 1u) ^ 1u, 200 + B_XFREE + 1)) return false;
    const int row = quad * 32 + lane;
    const int64_t tile = (int64_t)blockIdx.x + (int64_t)i * gridDim.x;
    const int64_t e = tile * ROWS + row;
    float x[K1];
#pragma unroll
    for (int k = 0; k < K1; ++k) x[k] = 0.f;
    if (e < p.n) {
        const float* src = p.obs + e * OBS;
        if (OBS % 4 == 0) {
#pragma unroll
            for (int k = 0; k < OBS / 4; ++k) {
                const float4 q = __ldcs(reinterpret_cast<const float4*>(src) + k);
                x[4 * k] = q.x; x[4 * k + 1] = q.y; x[4 * k + 2] = q.z; x[4 * k + 3] = q.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < OBS; ++k) x[k] = __ldcs(src + k);
        }
        const int64_t e_pf = e + (int64_t)3 * gridDim.x * ROWS;                 // the row this lane stages three tiles from now
        if (e_pf < p.n) {
            const char* nr = reinterpret_cast<const char*>(p.obs + e_pf * OBS);
            asm volatile("prefetch.global.L2 [%0];" ::"l"(nr));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(nr + OBS * 4 - 4));
        }
        if (p.norm) {
            const float* s_mean_hi = s_norm, * s_mean_lo = s_norm + 32, * s_istd = s_norm + 64;
#pragma unroll
            for (int k = 0; k < OBS; ++k) {
                // SB3 subtracts the float64 mean in float64; mean = hi + lo in float32 gives the same to ~2 ulp (qs_policy_tc.cu)
                const float v = __fmul_rn(__fadd_rn(__fadd_rn(x[k], -s_mean_hi[k]), -s_mean_lo[k]), s_istd[k]);
                x[k] = fminf(fmaxf(v, -p.norm_clip), p.norm_clip);
            }
        }
        if (p.obs_norm_out) {
            float* orow = p.obs_norm_out + e * OBS;
            if (OBS % 4 == 0) {
#pragma unroll
                for (int k = 0; k < OBS / 4; ++k) __stcs(reinterpret_cast<float4*>(orow) + k, make_float4(x[4 * k], x[4 * k + 1], x[4 * k + 2], x[4 * k + 3]));
            } else {
#pragma unroll
                for (int k = 0; k < OBS; ++k) __stcs(orow + k, x[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < OBS; ++k) x[k] = fminf(fmaxf(x[k], -60000.f), 60000.f);   // float16 range
    }
    x[OBS] = 1.0f;                                                       // multiplies the bias row of W1
    unsigned char* xt = smem + SM_X + xb * X_BYTES + row * 16;
#pragma unroll
    for (int kc = 0; kc < K1 / 8; ++kc) {
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) split_h2_rn(x[8 * kc + 2 * j], x[8 * kc + 2 * j + 1], h[j], l[j]);
        *reinterpret_cast<uint4*>(xt + kc * X_LBO) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(xt + X_HALF + kc * X_LBO) = make_uint4(l[0], l[1], l[2], l[3]);
    }
    fence_async_smem();                                                  // generic-proxy stores -> visible to the MMA (async proxy)
    __syncwarp();
    if (lane == 0) mbar_arrive(c.bar(B_XFULL + xb));
    return true;
}

template <int VER, bool FUSED>
__device__ __forceinline__ void role_env(const Ctx& c, const RoParams& p, int par, int quad, int lane, unsigned char* smem, const float* sC,
                                         const float4* s_mean, const float* s_val, unsigned long long noise_step) {
    // par: with ENV_SPLIT == 2 this warp serves the tiles of slot `par` only (local tiles i = par, par + 2, ...); else all tiles
    constexpr int OBS = EnvTraits<VER>::OBS;
    constexpr int STRIDE = ENV_SPLIT;                                   // tiles between two iterations of this warp
    const float* s_norm = reinterpret_cast<const float*>(smem + SM_NORM);
    float* tile_s = reinterpret_cast<float*>(smem + SM_TILE) + (par * 4 + quad) * 32 * 21;
    double* s_mom = reinterpret_cast<double*>(smem + SM_MOM) + (par * 4 + quad) * 40;
    const int row = quad * 32 + lane;
    const StepParams<float>& sp = p.sp;
    const bool moments = FUSED && sp.mom_partial != nullptr;
    double m1 = 0.0, m2 = 0.0, G = 0.0;
    if (moments && lane < OBS) {
        if (sp.mom_prev && sp.mom_prev[0] > 0.0) G = sp.mom_prev[1 + lane];
        else if (sp.mom_stats) G = sp.mom_stats[1 + lane];
    }
    const float ls[4] = {sC[C_LS], sC[C_LS + 1], sC[C_LS + 2], sC[C_LS + 3]};
    const float sd[4] = {__expf(ls[0]), __expf(ls[1]), __expf(ls[2]), __expf(ls[3])};
    const float lp0 = -(ls[0] + ls[1] + ls[2] + ls[3]) - 4.0f * 0.9189385332046727f;

    // the hidden state of the next tile: in registers one tile ahead when this warp is the only env warp of its scheduler (latency
    // it cannot hide otherwise); with two env warps per scheduler the record is only pulled into L2 ahead and loaded when needed
    constexpr bool REG_PREFETCH = ENV_SPLIT == 1;
    EnvState<float, VER> s_nx;
    if (FUSED && REG_PREFETCH) {
        const int64_t e0 = ((int64_t)blockIdx.x + (int64_t)par * gridDim.x) * ROWS + row;
        if (par < c.cnt && e0 < p.n) pool_load<float, VER>(sp.pool, sp.n, e0, s_nx);
    }
    // the X tile of local tile i + 2 is staged before tile i is stepped; the first iteration(s) only stage (one call site: code size)
    // With the deferred head (QS_RO_DEFER_HEAD) the outputs of a tile appear one job later, so this warp consumes them one of its
    // iterations later too (LAG): staging the X tile of a later tile must not queue behind the wait for them (measured: every
    // second job stalled ~4,000 cycles for its X tile otherwise).  The X buffers are released early (by the critic's layer-1 commit).
    constexpr int LAG = QS_RO_DEFER_HEAD ? STRIDE : 0;
    RO_TRACE_INIT();
#pragma unroll 1
    for (int j = par - 2; j < c.cnt + LAG; j += STRIDE) {
        RO_TRACE(0x300000u | (uint32_t)(j + 2));
        if (j + 2 < c.cnt && !stage_x<OBS>(c, p, j + 2, quad, lane, smem, s_norm)) return;
        RO_TRACE(0x310000u | (uint32_t)(j + 2));
        const int i = j - LAG;
        if (i < 0 || i >= c.cnt) continue;
        const int slot = i & 1;
        const uint32_t k = (uint32_t)i >> 1;
        const int64_t tile = (int64_t)blockIdx.x + (int64_t)i * gridDim.x;
        const int64_t e0 = tile * ROWS + quad * 32;
        const int64_t e = e0 + lane;
        const bool live = e < p.n;
        EnvState<float, VER> s;
        if (FUSED) {
            const int64_t en = e + (int64_t)STRIDE * gridDim.x * ROWS;
            if (REG_PREFETCH) {
                s = s_nx;
                if (i + STRIDE < c.cnt && en < p.n) pool_load<float, VER>(sp.pool, sp.n, en, s_nx);
            } else {
                if (live) pool_load<float, VER>(sp.pool, sp.n, e, s);
                if (i + STRIDE < c.cnt && en < p.n && lane < (PoolLayout<float, VER>::TILE_BYTES + 127) / 128)   // next tile record -> L2
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const unsigned char*>(sp.pool) + (en >> 5) * (int64_t)PoolLayout<float, VER>::TILE_BYTES + lane * 128));
            }
        }
        if (!(FUSED ? mbar_wait_bounded(c.bar(B_OUTF + slot * 4 + quad), k & 1u, 200 + B_OUTF + 1)
                    : mbar_wait_lazy(c.bar(B_OUTF + slot * 4 + quad), k & 1u, 200 + B_OUTF + 1))) return;
        RO_TRACE(0x320000u | (uint32_t)i);
        float4 mu = s_mean[slot * HEAD_SPLIT * ROWS + row];
        float value = s_val[slot * HEAD_SPLIT * ROWS + row];
#pragma unroll
        for (int hf = 1; hf < HEAD_SPLIT; ++hf) {                         // partial head sums of the other epilogue warp(s) of the row
            const float4 m2 = s_mean[(slot * HEAD_SPLIT + hf) * ROWS + row];
            mu.x += m2.x; mu.y += m2.y; mu.z += m2.z; mu.w += m2.w;
            value += s_val[(slot * HEAD_SPLIT + hf) * ROWS + row];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(c.bar(B_OUTE + slot * 4 + quad));
        float4 a = mu, ac = mu;
        if (live) {
            float4 eps = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.sample_mode == 1) eps = __ldcs(reinterpret_cast<const float4*>(p.noise) + e);
            else if (p.sample_mode == 2) eps = philox_normal4(p.noise_seed, (uint64_t)(sp.env_id_offset + e), noise_step);
            a.x = fmaf(sd[0], eps.x, mu.x); a.y = fmaf(sd[1], eps.y, mu.y); a.z = fmaf(sd[2], eps.z, mu.z); a.w = fmaf(sd[3], eps.w, mu.w);
            const float lp = fmaf(-0.5f, eps.x * eps.x + eps.y * eps.y + eps.z * eps.z + eps.w * eps.w, lp0);
            ac.x = fminf(fmaxf(a.x, p.lo[0]), p.hi[0]); ac.y = fminf(fmaxf(a.y, p.lo[1]), p.hi[1]);
            ac.z = fminf(fmaxf(a.z, p.lo[2]), p.hi[2]); ac.w = fminf(fmaxf(a.w, p.lo[3]), p.hi[3]);
            __stcs(reinterpret_cast<float4*>(p.actions) + e, a);
            if (p.actions_clipped) __stcs(reinterpret_cast<float4*>(p.actions_clipped) + e, ac);
            __stcs(p.values + e, value);
            __stcs(p.logp + e, lp);
        }
        if (FUSED) {
            float obs[OBS];
            if (live) {
                const float act[4] = {ac.x, ac.y, ac.z, ac.w};
                float Fcmd, Mcmd[3], F, M[3];
                scale_action<float>(sp.model, act, sp.scale_f32, Fcmd, Mcmd);
                mix_and_clamp<float>(sp.model, Fcmd, Mcmd, F, M);
                rk4_step_rolled<float>(sp.model, s.y, F, M, sp.substeps);
                renormalise_quat<float>(s.y);
                float reward;
                int ep_len;
                const uint32_t flags = step_logic<float, VER>(s, reward, ep_len);
                s.ep_ret += reward;
                make_obs<float, VER>(s, sp.obs_scaled, obs);
                sp.reward_out[e] = reward;
                sp.flags_out[e] = (uint8_t)flags;
                if (flags & (FLAG_TERMINATED | FLAG_TRUNCATED)) {
                    if (sp.term_obs_out) {
                        float* trow = sp.term_obs_out + e * OBS;
#pragma unroll
                        for (int q = 0; q < OBS; ++q) trow[q] = obs[q];
                    }
                    if (sp.ep_ret_out) sp.ep_ret_out[e] = s.ep_ret;
                    if (sp.ep_len_out) sp.ep_len_out[e] = ep_len;
                    if (sp.auto_reset) {
                        s.episode += 1;
                        reset_env<float, VER>(s, sp.rc, sp.seed, (uint64_t)(sp.env_id_offset + e));
                        make_obs<float, VER>(s, sp.obs_scaled, obs);
                    }
                }
                pool_store<float, VER>(sp.pool, sp.n, e, s);
#pragma unroll
                for (int q = 0; q < OBS; ++q) tile_s[lane * (OBS + 1) + q] = obs[q];
            }
            __syncwarp();
            const int64_t rem = p.n - e0;
            const int rows = rem < 32 ? (rem < 0 ? 0 : (int)rem) : 32;
            if (rows > 0) warp_store_rows<OBS>(sp.obs_out + e0 * OBS, tile_s, lane, rows);
            if (moments && lane < OBS && rows > 0) {
                const float L = tile_s[lane];
                double t1 = 0.0, t2 = 0.0;
#pragma unroll
                for (int r0 = 0; r0 < 32; r0 += 8) {
                    float a1 = 0.f, a2 = 0.f;
#pragma unroll
                    for (int r = r0; r < r0 + 8; ++r) {
                        const float v = r < rows ? tile_s[r * (OBS + 1) + lane] - L : 0.f;
                        a1 += v;
                        a2 = fmaf(v, v, a2);
                    }
                    t1 += (double)a1;
                    t2 += (double)a2;
                }
                const double dl = (double)L - G;
                m1 += t1 + (double)rows * dl;
                m2 += t2 + 2.0 * dl * t1 + (double)rows * dl * dl;
            }
            __syncwarp();
        }
    }
    if (moments && lane < OBS) { s_mom[lane] = m1; s_mom[OBS + lane] = m2; }
    RO_TRACE_END();
}

// ---------------------------------------------------------------------------------------------------------------------
// The kernel.
// ---------------------------------------------------------------------------------------------------------------------
template <int VER, bool FUSED>
__global__ void __launch_bounds__(RO_THREADS, 1) rollout_kernel(const RoParams p) {
    constexpr int OBS = EnvTraits<VER>::OBS;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float* sC = reinterpret_cast<float*>(smem + IMG_CONST);
    float4* s_mean = reinterpret_cast<float4*>(smem + SM_OUT_MEAN);
    float* s_val = reinterpret_cast<float*>(smem + SM_OUT_VAL);
    float* s_norm = reinterpret_cast<float*>(smem + SM_NORM);
    uint32_t* s_misc = reinterpret_cast<uint32_t*>(smem + SM_MISC);

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_misc)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 32) {
        const uint32_t b = smem_u32(smem + SM_BARS);
        for (int j = 0; j < N_BARS; ++j) {
            uint32_t count = 1u;                                                   // tcgen05.commit / one lane of one warp
            if ((j >= B_XFULL && j < B_XFULL + 3) || (j >= B_H1 && j < B_D3FREE)) count = 4u;   // one arrival per quadrant warp
            if (j >= B_D3FREE && j < B_D3FREE + 2) count = 4u * HEAD_SPLIT;         // every epilogue warp of the slot that reads D3
            if (j >= B_OUTF && j < B_OUTF + 8) count = HEAD_SPLIT;
            tc::mbar_init(b + 8u * j, count);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // operand image -> shared memory (prepared once per parameter update by policy_prepare_kernel), or staged from the raw blob
    if (p.image) {
        const uint4* src = reinterpret_cast<const uint4*>(p.image);
        uint4* dst = reinterpret_cast<uint4*>(smem);
        for (int j = tid; j < IMG_BYTES / 16; j += RO_THREADS) dst[j] = __ldg(src + j);
    } else {
        const Blob B{OBS};
        for (int net = 0; net < 2; ++net) {
            const float sc = 2.8853900817779268f;                  // 2 log2(e): accumulators come out as exponents of 2
            stage_weights<true, RO_THREADS>(p.params + B.w1(net), p.params + B.b1(net), OBS, OBS, K1, N1, sc, smem + IMG_WHI + OFF_W1 + net * W1_BYTES,
                                            smem + IMG_WLO + OFF_W1 + net * W1_BYTES, tid);
            stage_weights<true, RO_THREADS>(p.params + B.w2(net), p.params + B.b2(net), N1, N1, N1 + KB, N2, sc, smem + IMG_WHI + OFF_W2 + net * W2_BYTES,
                                            smem + IMG_WLO + OFF_W2 + net * W2_BYTES, tid);
            stage_weights<true, RO_THREADS>(p.params + B.w3(net), p.params + B.b3(net), N2, N2, N2 + KB, N3, sc, smem + IMG_WHI + OFF_W3 + net * W3_BYTES,
                                            smem + IMG_WLO + OFF_W3 + net * W3_BYTES, tid);
            for (int j = tid; j < N3 * NACT; j += RO_THREADS) sC[C_WH + net * N3 * NACT + j] = __ldg(p.params + B.wh(net) + j);
            if (tid < NACT) sC[C_BH + net * NACT + tid] = __ldg(p.params + B.bh(net) + tid);
        }
        if (tid < NACT) sC[C_LS + tid] = __ldg(p.params + B.log_std() + tid);
    }
    // the constant A tile of the bias k-steps: row r = (1, 0, ..., 0)
    for (int j = tid; j < ONE_BYTES / 16; j += RO_THREADS)
        reinterpret_cast<uint4*>(smem + SM_ONE)[j] = j < ROWS ? make_uint4(0x00003C00u, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
    if (tid < 32) {
        double m = 0.0, is = 1.0;
        if (p.norm && tid < OBS) {
            m = p.norm[1 + tid];
            is = 1.0 / sqrt(p.norm[1 + OBS + tid] + (double)p.norm_eps);
        }
        s_norm[tid] = (float)m;
        s_norm[32 + tid] = (float)(m - (double)(float)m);
        s_norm[64 + tid] = (float)is;
    }
    unsigned long long noise_step = 0;
    if (p.sample_mode == 2 && p.noise_step) noise_step = *reinterpret_cast<const volatile unsigned long long*>(p.noise_step);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    Ctx c;
    c.sbase = smem_u32(smem);
    c.tmem = s_misc[0];
    const int64_t n_tiles = (p.n + ROWS - 1) / ROWS;
    c.cnt = (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);

    if (warp >= W_EPI0 && warp < W_EPI0 + EPI_WARPS) {
        if (REBALANCE && REGS_EPI > REGS_LAUNCH) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
        if (REBALANCE && REGS_EPI < REGS_LAUNCH) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
        role_epilogue(c, (warp - W_EPI0) / (4 * EPI_SPLIT), ((warp - W_EPI0) >> 2) % EPI_SPLIT, warp & 3, lane, sC, s_mean, s_val);
        if (REBALANCE && REGS_EPI > REGS_LAUNCH) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LAUNCH));
        if (REBALANCE && REGS_EPI < REGS_LAUNCH) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_LAUNCH));
    } else if (warp >= W_ENV0 && warp < W_ENV0 + ENV_WARPS) {
        if (REBALANCE) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_ENV));
        role_env<VER, FUSED>(c, p, ENV_SPLIT == 2 ? (warp - W_ENV0) >> 2 : 0, warp & 3, lane, smem, sC, s_mean, s_val, noise_step);
        if (REBALANCE) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_LAUNCH));
    } else {
        if (REBALANCE) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_MMA));
        if (warp < W_MMA0 + MMA_WARPS) role_mma(c, warp - W_MMA0);
        if (REBALANCE) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_LAUNCH));   // the common tail runs at the launch value again
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(c.tmem), "r"(TMEM_COLS));
    }
    if (!FUSED) {
        // in-kernel sampling without the env step: the last CTA to finish advances the device step counter (ticket = counter[1])
        if (p.sample_mode == 2 && p.noise_step) {
            __threadfence();
            __syncthreads();
            if (tid == 0) s_misc[1] = atomicAdd(p.ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
            __syncthreads();
            if (s_misc[1] != 0u && tid == 0) {
                *p.ticket = 0u;
                *p.noise_step = noise_step + 1ull;
            }
        }
        return;
    }

    // ---- per-CTA moment partials, then the LAST CTA to finish: fixed-order sum of the partials -> (n, mean, M2) -> Chan merge
    const StepParams<float>& sp = p.sp;
    const bool moments = sp.mom_partial != nullptr;
    if (moments && tid < 2 * OBS) {
        const double* sm = reinterpret_cast<const double*>(smem + SM_MOM);
        double a = 0.0;
#pragma unroll
        for (int w = 0; w < ENV_WARPS; ++w) a += sm[w * 40 + tid];
        sp.mom_partial[(int64_t)blockIdx.x * 2 * OBS + tid] = a;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_misc[1] = atomicAdd(p.ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if (s_misc[1] == 0u) return;
    __threadfence();
    if (tid == 0) {
        *p.ticket = 0u;
        if (p.sample_mode == 2 && p.noise_step) *p.noise_step = noise_step + 1ull;
    }
    if (!moments) return;
    double* red = reinterpret_cast<double*>(smem);                  // the operand image is dead: [slices][2 * OBS] scratch
    constexpr int W2 = 2 * OBS, SL = RO_THREADS / W2;
    const int col = tid % W2, slice = tid / W2;
    double shift = 0.0;
    if (tid < OBS) shift = p.mom_out[0] > 0.0 ? p.mom_out[1 + tid] : (sp.mom_stats ? sp.mom_stats[1 + tid] : 0.0);   // the offset rule of role_env
    if (slice < SL) {
        double acc = 0.0;
        for (int b = slice; b < (int)gridDim.x; b += SL) acc += __ldcg(sp.mom_partial + (int64_t)b * W2 + col);
        red[slice * W2 + col] = acc;
    }
    __syncthreads();
    const double cnt = (double)p.n;
    double mean_b = 0.0, m2_b = 0.0, count = 0.0, mean_r = 0.0, var_r = 0.0;
    if (tid < OBS) {
        double s1 = 0.0, s2 = 0.0;
        for (int k = 0; k < SL; ++k) { s1 += red[k * W2 + tid]; s2 += red[k * W2 + OBS + tid]; }
        mean_b = shift + s1 / cnt;
        m2_b = s2 - s1 * s1 / cnt;
        if (p.mom_merge) {
            count = p.mom_merge[0]; mean_r = p.mom_merge[1 + tid]; var_r = p.mom_merge[1 + OBS + tid];
            const double delta = mean_b - mean_r, tot = count + cnt;
            mean_r = mean_r + delta * cnt / tot;
            var_r = (var_r * count + m2_b + delta * delta * count * cnt / tot) / tot;
            count = tot;
        }
    }
    __syncthreads();                                                  // every column has read the old triplet / count
    if (tid < OBS) {
        p.mom_out[1 + tid] = mean_b;
        p.mom_out[1 + OBS + tid] = m2_b;
        if (tid == 0) p.mom_out[0] = cnt;
        if (p.mom_merge) {
            p.mom_merge[1 + tid] = mean_r;
            p.mom_merge[1 + OBS + tid] = var_r;
            if (tid == 0) p.mom_merge[0] = count;
        }
    }
}

// raw float32 blob -> the operand image (float16 hi / lo canonical B operands, pre-scaled by 2 log2 e, + the float32 head)
template <int OBS>
__global__ void __launch_bounds__(256) policy_prepare_kernel(const float* __restrict__ params, unsigned char* __restrict__ image) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    constexpr int NT = 256 * 8;
    const Blob B{OBS};
    float* sC = reinterpret_cast<float*>(image + IMG_CONST);
    for (int net = 0; net < 2; ++net) {
        const float sc = 2.8853900817779268f;
        stage_weights<true, NT>(params + B.w1(net), params + B.b1(net), OBS, OBS, K1, N1, sc, image + IMG_WHI + OFF_W1 + net * W1_BYTES,
                                image + IMG_WLO + OFF_W1 + net * W1_BYTES, tid);
        stage_weights<true, NT>(params + B.w2(net), params + B.b2(net), N1, N1, N1 + KB, N2, sc, image + IMG_WHI + OFF_W2 + net * W2_BYTES,
                                image + IMG_WLO + OFF_W2 + net * W2_BYTES, tid);
        stage_weights<true, NT>(params + B.w3(net), params + B.b3(net), N2, N2, N2 + KB, N3, sc, image + IMG_WHI + OFF_W3 + net * W3_BYTES,
                                image + IMG_WLO + OFF_W3 + net * W3_BYTES, tid);
        for (int j = tid; j < N3 * NACT; j += NT) sC[C_WH + net * N3 * NACT + j] = params[B.wh(net) + j];
        if (tid < NACT) sC[C_BH + net * NACT + tid] = params[B.bh(net) + tid];
    }
    if (tid < NACT) sC[C_LS + tid] = params[B.log_std() + tid];
}

template <int VER, bool FUSED>
static cudaError_t launch(const RoParams& p, int sms, cudaStream_t st) {
    auto k = rollout_kernel<VER, FUSED>;
    cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL);
    if (err != cudaSuccess) return err;
    const int64_t tiles = (p.n + ROWS - 1) / ROWS;
    const unsigned grid = (unsigned)(tiles < sms ? tiles : sms);
    k<<<grid, RO_THREADS, SM_TOTAL, st>>>(p);
    return cudaGetLastError();
}

}  // namespace QS_RO_NS

#ifdef QS_RO_BUILD_POLICY
// the policy forward alone through the warp-specialised pipeline (QS_POLICY_TENSOR of qs_policy_forward)
int launch_policy_pipeline(const float* params, int obs_dim, const float* obs, const float* noise, int64_t n, const double* norm_stats,
                           float norm_eps, float norm_clip, float* obs_norm_out, float* actions, float* actions_clipped,
                           const float* clip_lo, const float* clip_hi, float* values, float* logp, cudaStream_t stream,
                           const char** err_out, uint64_t philox_seed, uint64_t* philox_counter, int64_t env_id_offset) {
    static thread_local char msg[256];
    QS_RO_NS::RoParams p;
    memset(&p, 0, sizeof(p));
    p.params = params; p.obs = obs; p.norm = norm_stats; p.norm_eps = norm_eps; p.norm_clip = norm_clip;
    p.sample_mode = noise ? 1 : 0; p.noise = noise;
    if (philox_counter) {             // in-kernel Gaussian noise: counter[0] = step (advanced by the kernel), counter[1] = last-CTA ticket
        p.sample_mode = 2; p.noise = nullptr; p.noise_seed = philox_seed;
        p.noise_step = reinterpret_cast<unsigned long long*>(philox_counter);
        p.ticket = reinterpret_cast<unsigned int*>(philox_counter + 1);
        p.sp.env_id_offset = env_id_offset;
    }
    for (int i = 0; i < 4; ++i) { p.lo[i] = clip_lo ? clip_lo[i] : -3.4e38f; p.hi[i] = clip_hi ? clip_hi[i] : 3.4e38f; }
    p.obs_norm_out = obs_norm_out; p.actions = actions; p.actions_clipped = actions_clipped; p.values = values; p.logp = logp; p.n = n;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const cudaError_t err = obs_dim == 20 ? QS_RO_NS::launch<ENV_V2, false>(p, sms, stream) : QS_RO_NS::launch<ENV_V1, false>(p, sms, stream);
    if (err != cudaSuccess) {
        snprintf(msg, sizeof(msg), "rollout_kernel<policy only>: %s", cudaGetErrorString(err));
        *err_out = msg;
        return QS_ECUDA;
    }
    return QS_OK;
}


// sticky status of the policy-part kernels (read and cleared; see qs_rollout_status)
int policy_pipeline_status() {
    int v = 0;
    if (cudaMemcpyFromSymbol(&v, QS_RO_NS::g_ro_status, sizeof(int)) != cudaSuccess) return -1;
    if (v != 0) {
        const int zero = 0;
        cudaMemcpyToSymbol(QS_RO_NS::g_ro_status, &zero, sizeof(int));
    }
    return v;
}
#endif  // QS_RO_BUILD_POLICY
}  // namespace qs
#ifdef QS_RO_TRACE
#ifdef QS_RO_BUILD_POLICY
extern "C" int qs_trace_dump_policy(void* out, int bytes) {
#else
extern "C" int qs_trace_dump_fused(void* out, int bytes) {
#endif
    cudaDeviceSynchronize();
    return (int)cudaMemcpyFromSymbol(out, qs::QS_RO_NS::g_ro_trace, bytes < (int)sizeof(qs::QS_RO_NS::g_ro_trace) ? bytes : sizeof(qs::QS_RO_NS::g_ro_trace));
}
#endif
namespace qs {

#ifdef QS_RO_BUILD_FUSED
int policy_pipeline_status();
#endif
}  // namespace qs

#ifdef QS_RO_BUILD_FUSED
using namespace qs;

extern "C" {

int64_t qs_policy_image_bytes(void) { return QS_RO_NS::IMG_BYTES; }

int qs_policy_prepare(const float* params, int obs_dim, void* image_out, void* stream) {
    if (!params || !image_out || (obs_dim != 20 && obs_dim != 17)) { set_error(nullptr, "qs_policy_prepare: bad argument (obs_dim 17 or 20)"); return QS_EINVAL; }
    if (reinterpret_cast<uintptr_t>(image_out) & 15) { set_error(nullptr, "qs_policy_prepare: image_out must be 16-byte aligned"); return QS_EINVAL; }
    cudaMemsetAsync(image_out, 0, QS_RO_NS::IMG_BYTES, (cudaStream_t)stream);
    if (obs_dim == 20) QS_RO_NS::policy_prepare_kernel<20><<<8, 256, 0, (cudaStream_t)stream>>>(params, (unsigned char*)image_out);
    else QS_RO_NS::policy_prepare_kernel<17><<<8, 256, 0, (cudaStream_t)stream>>>(params, (unsigned char*)image_out);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) { set_error(nullptr, "qs_policy_prepare: %s", cudaGetErrorString(err)); return QS_ECUDA; }
    return QS_OK;
}

int qs_rollout_step(qs_handle* h, const qs_rollout_args* a, void* stream) {
    if (!h || !a) { set_error(h, "qs_rollout_step: null argument"); return QS_EINVAL; }
    if (h->cfg.precision != QS_F32 || h->cfg.integrator != QS_RK4) { set_error(h, "qs_rollout_step: float32 / RK4 handles only"); return QS_EINVAL; }
    if (!h->initialized) { set_error(h, "qs_rollout_step: call qs_reset first"); return QS_EINVAL; }
    if (h->dyn_on) { set_error(h, "qs_rollout_step: the fused rollout kernel has no dynamics randomisation; use qs_policy_forward + qs_step, or disarm qs_dynamics_randomization"); return QS_EINVAL; }
    if (!a->policy_image || !a->obs || !a->obs_next || !a->actions_out || !a->values_out || !a->logp_out || !a->reward_out || !a->flags_out) {
        set_error(h, "qs_rollout_step: policy_image, obs, obs_next, actions_out, values_out, logp_out, reward_out and flags_out are required");
        return QS_EINVAL;
    }
    if (a->sample_mode < QS_SAMPLE_MEAN || a->sample_mode > QS_SAMPLE_PHILOX || (a->sample_mode == QS_SAMPLE_NOISE && !a->noise) ||
        (a->sample_mode == QS_SAMPLE_PHILOX && !a->noise_step)) {
        set_error(h, "qs_rollout_step: sample_mode needs its noise buffer (QS_SAMPLE_NOISE) or device step counter (QS_SAMPLE_PHILOX)");
        return QS_EINVAL;
    }
    const uintptr_t al = reinterpret_cast<uintptr_t>(a->policy_image) | reinterpret_cast<uintptr_t>(a->actions_out) | reinterpret_cast<uintptr_t>(a->noise) |
                         reinterpret_cast<uintptr_t>(a->actions_clipped_out) | reinterpret_cast<uintptr_t>(a->obs) | reinterpret_cast<uintptr_t>(a->obs_next) |
                         reinterpret_cast<uintptr_t>(a->obs_norm_out);
    if (al & 15) { set_error(h, "qs_rollout_step: image, obs, noise and action buffers must be 16-byte aligned"); return QS_EINVAL; }
    cudaError_t err = cudaSetDevice(h->cfg.device);
    if (err != cudaSuccess) { set_error(h, "qs_rollout_step: cudaSetDevice: %s", cudaGetErrorString(err)); return QS_ECUDA; }
    if (!h->ro_ticket) {
        err = cudaMalloc(&h->ro_ticket, sizeof(unsigned int));
        if (err == cudaSuccess) err = cudaMemset(h->ro_ticket, 0, sizeof(unsigned int));
        if (err != cudaSuccess) { set_error(h, "qs_rollout_step: ticket allocation: %s", cudaGetErrorString(err)); return QS_ECUDA; }
    }
    QS_RO_NS::RoParams p;
    memset(&p, 0, sizeof(p));
    p.image = static_cast<const unsigned char*>(a->policy_image);
    p.obs = a->obs; p.norm = a->norm_stats; p.norm_eps = a->norm_eps; p.norm_clip = a->norm_clip;
    p.sample_mode = a->sample_mode; p.noise = a->noise; p.noise_seed = a->noise_seed;
    p.noise_step = reinterpret_cast<unsigned long long*>(a->noise_step);
    for (int i = 0; i < 4; ++i) { p.lo[i] = a->clip_lo[i]; p.hi[i] = a->clip_hi[i]; }
    p.obs_norm_out = a->obs_norm_out; p.actions = a->actions_out; p.actions_clipped = a->actions_clipped_out;
    p.values = a->values_out; p.logp = a->logp_out; p.n = h->cfg.n_envs;
    p.sp = base_params<float>(h);
    p.sp.actions = nullptr;
    p.sp.obs_out = a->obs_next; p.sp.reward_out = a->reward_out; p.sp.flags_out = a->flags_out;
    p.sp.term_obs_out = a->terminal_obs_out; p.sp.ep_ret_out = a->ep_return_out; p.sp.ep_len_out = a->ep_len_out;
    p.sp.ls_counters = nullptr; p.sp.ls_steps = nullptr;
    p.mom_out = h->mom_out; p.mom_merge = h->mom_merge; p.ticket = h->ro_ticket;
    QS_FOR_VARIANT(h, err = (QS_RO_NS::launch<VER, true>(p, h->num_sms, (cudaStream_t)stream)););
    if (err != cudaSuccess) { set_error(h, "rollout_kernel launch failed: %s", cudaGetErrorString(err)); return QS_ECUDA; }
    return QS_OK;
}

int qs_rollout_status(void) {
    int v = 0, w = qs::policy_pipeline_status();
    if (cudaMemcpyFromSymbol(&v, QS_RO_NS::g_ro_status, sizeof(int)) != cudaSuccess) return -1;
    if (v != 0) {
        const int zero = 0;
        cudaMemcpyToSymbol(QS_RO_NS::g_ro_status, &zero, sizeof(int));
    }
    return v != 0 ? v : w;
}

}  // extern "C"

#endif  // QS_RO_BUILD_FUSED
