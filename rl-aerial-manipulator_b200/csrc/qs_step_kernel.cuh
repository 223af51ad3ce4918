// qs_step_kernel.cuh -- the fused env-step kernel: one thread per env, hidden state in registers.
//
//   load state (LDG.128 planes) + action (LDG.128)
//   -> action scaling, mixer, per-prop clamp            [quadcopter.py:105-112]
//   -> integrator: RK4 x substeps, or the LSODA port     [quadcopter.py:113]
//   -> quaternion renormalisation                        [quadcopter.py:114]
//   -> reward + waypoint/hold/termination state machine  [rl_env_scaledObs.py step/_calculate_reward]
//   -> observation (scaled, float32)                     [_get_observation]
//   -> auto-reset with Philox draws for done envs        [DummyVecEnv.step_wait + reset()]
//   -> store state planes; obs rows leave through a per-warp shared-memory transpose so the
//      [n, obs_dim] row-major output is written with full 128-bit coalesced stores.
//   -> optionally, VecNormalize's batch moments of the returned observations: lane c of each warp adds column c of
//      the warp's shared-memory obs tile in float64 (conflict-free: row stride OBS+1), CTA partials are combined
//      in shared memory and written once per CTA -- the separate 34 us read pass over the obs disappears.
#pragma once
#include "qs_pool.cuh"
#include "qs_lsoda.cuh"

namespace qs {

enum : int { INTEG_RK4 = 0, INTEG_LSODA = 1 };

template <typename Real>
struct StepParams {
    void* pool;
    int64_t n;
    const float* actions;       // [n,4]
    float* obs_out;             // [n,OBS]
    Real* reward_out;           // [n]
    uint8_t* flags_out;         // [n]
    float* term_obs_out;        // [n,OBS] or null
    Real* ep_ret_out;           // [n] or null
    int32_t* ep_len_out;        // [n] or null
    const LsodaTables* ls_tables; // device copy of the method coefficients (LSODA mode)
    double* mom_partial;        // [gridDim.x][2*OBS] per-CTA column sums of (obs - shift), (obs - shift)^2, or null
    const double* mom_stats;    // VecNormalize stats (count, mean[OBS], var[OBS]) or null
    const double* mom_prev;     // the previous step's triplet (n, mean, M2): its mean is the summation offset G when n > 0,
                                // else the running mean of mom_stats, else 0 (moments_final_kernel applies the same rule)
    int32_t* ls_counters;       // [n,4] or null (LSODA diagnostics)
    double* ls_steps;           // [n,2] or null
    int substeps, obs_scaled, scale_f32, auto_reset;
    uint64_t seed;
    int64_t env_id_offset;
    double rtol, atol;
    Model<Real> model;
    ResetConsts rc;
    Real* dyn;                  // dynamics randomisation: planes [N_DYN][dyn_stride] (k_m, k_I, eta[4], f_wind[3]), or null = off
    int64_t dyn_stride;
    DynRand dr;                 // ... and how a reset draws them
    int64_t pad_;               // 64 bytes appended in all: the fields of ManyParams behind it keep their 16-byte alignment, and the
                                // nominal qs_step_many kernels their constant loads
};

// One env's parameters: N_DYN coalesced plane reads; a reset draws the new episode's and stores them.
template <typename Real>
QS_HD void dyn_load(const StepParams<Real>& p, int64_t e, Real* d) {
#pragma unroll
    for (int k = 0; k < N_DYN; ++k) d[k] = p.dyn[k * p.dyn_stride + e];
}
template <typename Real>
QS_HD void dyn_redraw(Real* planes, int64_t stride, const DynRand& r, uint64_t env_gid, uint32_t episode, int64_t e, Real* d) {
    double v[N_DYN];
    dyn_draw(r, env_gid, episode, v);
#pragma unroll
    for (int k = 0; k < N_DYN; ++k) {
        d[k] = (Real)v[k];
        planes[k * stride + e] = d[k];
    }
}

#if defined(__CUDACC__)
constexpr int STEP_BLOCK = 128;
// resident CTAs per SM the float32/RK4 kernel is compiled for (caps registers at 65536/(128*N)) and whether it prefetches
// the next tile into registers.  Measured on B200, 1M envs (profiles/r01/README.md): no prefetch 4/5/6/8 CTAs: 64.5 / 58.0 /
// 65.2 / 72.4 us; prefetch 2/3/4/5 CTAs: 62.2 / 54.6 / 60.0 / 68.9 us (5: spills).  The kernel is half issue (~26 us of
// instructions per SM), half HBM latency: what it needs is loads in flight, not resident warps.
// float64 and LSODA need the registers more than the occupancy.
#ifndef QS_STEP_MINB_F32
#define QS_STEP_MINB_F32 3
#endif
#ifndef QS_STEP_PREFETCH_F32
#define QS_STEP_PREFETCH_F32 1
#endif
template <typename Real, int INTEG> struct StepOcc { static constexpr int MINB = 1; static constexpr bool PREFETCH = false; };
#ifndef QS_STEP_MINB_F64
#define QS_STEP_MINB_F64 3
#endif
#ifndef QS_STEP_PREFETCH_F64
#define QS_STEP_PREFETCH_F64 0
#endif
template <> struct StepOcc<double, 0> { static constexpr int MINB = QS_STEP_MINB_F64; static constexpr bool PREFETCH = QS_STEP_PREFETCH_F64 != 0; };
template <> struct StepOcc<float, 0> { static constexpr int MINB = QS_STEP_MINB_F32; static constexpr bool PREFETCH = QS_STEP_PREFETCH_F32 != 0; };

// Row-major [32, OBS] tile of one warp -> global, 128 bits per lane per store.
template <int OBS>
__device__ __forceinline__ void warp_store_rows(float* __restrict__ dst, const float* tile /*[32][OBS+1]*/, int lane, int valid_rows) {
    constexpr int TOTAL = 32 * OBS;
    const int valid = valid_rows * OBS;
#pragma unroll
    for (int base = 0; base < TOTAL; base += 128) {
        const int e = base + 4 * lane;
        if (e + 3 < valid) {
            float4 v;
            v.x = tile[((e + 0) / OBS) * (OBS + 1) + (e + 0) % OBS];
            v.y = tile[((e + 1) / OBS) * (OBS + 1) + (e + 1) % OBS];
            v.z = tile[((e + 2) / OBS) * (OBS + 1) + (e + 2) % OBS];
            v.w = tile[((e + 3) / OBS) * (OBS + 1) + (e + 3) % OBS];
            __stcs(reinterpret_cast<float4*>(dst + e), v);
        } else {
            for (int j = 0; j < 4; ++j)
                if (e + j < valid) dst[e + j] = tile[((e + j) / OBS) * (OBS + 1) + (e + j) % OBS];
        }
    }
}

// DYN: dynamics randomisation (RK4 only) -- the env's parameters are read from p.dyn every step and redrawn at an auto-reset.
template <typename Real, int VER, int INTEG, bool MOMENTS = false, bool DYN = false>
__global__ void __launch_bounds__(STEP_BLOCK, StepOcc<Real, INTEG>::MINB) env_step_kernel(const StepParams<Real> p) {
    static_assert(!DYN || INTEG == INTEG_RK4, "dynamics randomisation is RK4 only");
    constexpr int OBS = EnvTraits<VER>::OBS;
    __shared__ float s_tile[STEP_BLOCK / 32][32 * (OBS + 1)];
    __shared__ double s_mom[MOMENTS ? STEP_BLOCK / 32 : 1][2 * OBS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double m1 = 0.0, m2 = 0.0;                       // lane c < OBS: running sums of column c over this warp's tiles
    double G = 0.0;
    if (MOMENTS && lane < OBS) {
        if (p.mom_prev && p.mom_prev[0] > 0.0) G = p.mom_prev[1 + lane];
        else if (p.mom_stats) G = p.mom_stats[1 + lane];
    }
    const int64_t warps_total = (int64_t)gridDim.x * (STEP_BLOCK / 32);
    const int64_t n_warp_tiles = (p.n + 31) / 32;
    float* tile = s_tile[warp];

    // software prefetch (float32/RK4 only): the state and action of this warp's NEXT tile are requested before the current
    // tile is integrated, so every resident warp always has ~100 B per lane in flight instead of loading, then computing
    constexpr bool PREFETCH = StepOcc<Real, INTEG>::PREFETCH;
    EnvState<Real, VER> s_nx;
    float4 a_nx = make_float4(0.f, 0.f, 0.f, 0.f);
    int64_t wt = (int64_t)blockIdx.x * (STEP_BLOCK / 32) + warp;
    if (PREFETCH && wt < n_warp_tiles && wt * 32 + lane < p.n) {
        pool_load<Real, VER>(p.pool, p.n, wt * 32 + lane, s_nx);
        a_nx = __ldcs(reinterpret_cast<const float4*>(p.actions) + wt * 32 + lane);
    }
    for (; wt < n_warp_tiles; wt += warps_total) {
        const int64_t e0 = wt * 32;
        const int64_t e = e0 + lane;
        const bool live = e < p.n;
        float obs[OBS];
        EnvState<Real, VER> s;
        float4 a4;
        if (PREFETCH) {
            s = s_nx;
            a4 = a_nx;
            const int64_t en = (wt + warps_total) * 32 + lane;
            if (wt + warps_total < n_warp_tiles && en < p.n) {
                pool_load<Real, VER>(p.pool, p.n, en, s_nx);
                a_nx = __ldcs(reinterpret_cast<const float4*>(p.actions) + en);
            }
        }
        if constexpr (DYN) {
            // the next tile's parameter planes are pulled into L2 (no registers held): their loads then wait on L2, not HBM
            constexpr int LINES = (int)sizeof(Real) * 32 / 128;
            const int64_t wn = wt + warps_total;
            if (wn < n_warp_tiles && lane < N_DYN * LINES)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(p.dyn + (lane / LINES) * p.dyn_stride + wn * 32 + (lane % LINES) * (128 / (int)sizeof(Real))));
        }
#ifdef QS_STEP_L2_PREFETCH          // A/B: no register prefetch, but the next tile's record and actions are pulled into L2
        if (!PREFETCH) {
            using L = PoolLayout<Real, VER>;
            const int64_t wn = wt + warps_total;
            if (wn < n_warp_tiles) {
                constexpr int LINES = (L::TILE_BYTES + 127) / 128;
                const unsigned char* rec = reinterpret_cast<const unsigned char*>(p.pool) + wn * (int64_t)L::TILE_BYTES;
                for (int l = lane; l < LINES; l += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(rec + l * 128));
                if (lane < 4) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const unsigned char*>(p.actions + wn * 128) + lane * 128));
            }
        }
#endif
        if (live) {
            if (!PREFETCH) {
                pool_load<Real, VER>(p.pool, p.n, e, s);
                a4 = __ldcs(reinterpret_cast<const float4*>(p.actions) + e);
            }
            const float act[4] = {a4.x, a4.y, a4.z, a4.w};

            Real Fcmd, Mcmd[3], F, M[3];
            scale_action<Real>(p.model, act, p.scale_f32, Fcmd, Mcmd);
            uint32_t flags = 0;
            if constexpr (DYN) {
                Real d[N_DYN], aw[3];
                dyn_load(p, e, d);
                dyn_forces<Real>(p.model, Fcmd, Mcmd, d, F, M, aw);
                rk4_step<Real, true>(p.model, s.y, F, M, p.substeps, aw);
            } else if constexpr (INTEG == INTEG_LSODA) {
                mix_and_clamp<Real>(p.model, Fcmd, Mcmd, F, M);
                LsodaResult r;
                lsoda_advance(p.model, *p.ls_tables, s.y, F, M, p.model.dt, p.rtol, p.atol, r);
                if (r.status & ~LS_WOULD_SWITCH) flags |= FLAG_LSODA_FAIL;
                if (p.ls_counters) {
                    reinterpret_cast<int4*>(p.ls_counters)[e] = make_int4(r.nst, r.nfe, r.nqu, r.status);
                    reinterpret_cast<double2*>(p.ls_steps)[e] = make_double2(r.hu, r.tcur);
                }
            } else {
                mix_and_clamp<Real>(p.model, Fcmd, Mcmd, F, M);
                rk4_step<Real>(p.model, s.y, F, M, p.substeps);
            }
            renormalise_quat<Real>(s.y);

            Real reward;
            int ep_len;
            flags |= step_logic<Real, VER>(s, reward, ep_len);
            s.ep_ret += reward;
            make_obs<Real, VER>(s, p.obs_scaled, obs);

            p.reward_out[e] = reward;
            p.flags_out[e] = (uint8_t)flags;
            if (flags & (FLAG_TERMINATED | FLAG_TRUNCATED)) {
                if (p.term_obs_out) {
                    float* row = p.term_obs_out + e * OBS;
#pragma unroll
                    for (int i = 0; i < OBS; ++i) row[i] = obs[i];
                }
                if (p.ep_ret_out) p.ep_ret_out[e] = s.ep_ret;
                if (p.ep_len_out) p.ep_len_out[e] = ep_len;
                if (p.auto_reset) {
                    s.episode += 1;
                    reset_env<Real, VER>(s, p.rc, p.seed, (uint64_t)(p.env_id_offset + e));
                    make_obs<Real, VER>(s, p.obs_scaled, obs);
                    if constexpr (DYN) {
                        Real d[N_DYN];
                        dyn_redraw(p.dyn, p.dyn_stride, p.dr, (uint64_t)(p.env_id_offset + e), s.episode, e, d);
                    }
                }
            }
            pool_store<Real, VER>(p.pool, p.n, e, s);
#pragma unroll
            for (int i = 0; i < OBS; ++i) tile[lane * (OBS + 1) + i] = obs[i];
        }
        __syncwarp();
        const int64_t rem = p.n - e0;
        const int rows = rem < 32 ? (int)rem : 32;
        warp_store_rows<OBS>(p.obs_out + e0 * OBS, tile, lane, rows);
        if (MOMENTS && lane < OBS) {
            // float32 sums over 8 rows of (obs - L), L = the tile's first row (deviations ~ one sigma: always well conditioned),
            // re-centred to the global offset G in float64 once per tile:  sum(x-G) = sum(x-L) + k(L-G), and the square likewise
            const float L = tile[lane];
            double t1 = 0.0, t2 = 0.0;
#pragma unroll
            for (int r0 = 0; r0 < 32; r0 += 8) {
                float a1 = 0.f, a2 = 0.f;
#pragma unroll
                for (int r = r0; r < r0 + 8; ++r) {
                    const float v = r < rows ? tile[r * (OBS + 1) + lane] - L : 0.f;
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
    if (MOMENTS) {
        if (lane < OBS) { s_mom[warp][lane] = m1; s_mom[warp][OBS + lane] = m2; }
        __syncthreads();
        if (threadIdx.x < 2 * OBS) {
            double a = 0.0;
#pragma unroll
            for (int w = 0; w < STEP_BLOCK / 32; ++w) a += s_mom[w][threadIdx.x];
            p.mom_partial[(int64_t)blockIdx.x * 2 * OBS + threadIdx.x] = a;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// float32 / RK4 throughput kernel with a TMA-fed shared-memory pipeline.
//
// Same per-env body as env_step_kernel, but the hidden state and the action of a warp tile (32 envs: NVEC x 512 B planes,
// the tail plane, 512 B of actions) are brought in by cp.async.bulk (UBLKCP) into a per-warp ring of STAGES tiles, each
// guarded by its own mbarrier.  The copies of the next STAGES-1 tiles are always in flight while the current one is
// integrated, without holding them in registers -- env_step_kernel needs ~100 B per lane in flight to cover the ~1 us HBM
// latency and measured 0.74 of the copy bandwidth; register double-buffering got 0.79 at 159 registers.
//
// MEASURED SLOWER than the register-prefetch kernel (1M envs: 2 stages x 4/5/6 CTAs = 61.5 / 62.7 / 65.7 us vs 54.6 us): seven
// 512-byte bulk copies per tile issued by one lane, an mbarrier wait and a shared-memory round trip cost more than they
// hide.  Kept as an opt-in (QS_STEP_F32_TMA=1) with its own parity test so the comparison stays reproducible.
// ------------------------------------------------------------------------------------------------------------------
#ifndef QS_TMA_STAGES
#define QS_TMA_STAGES 2
#endif
constexpr int TMA_STAGES = QS_TMA_STAGES;   // tiles in flight per warp (incl. the current one); A/B in profiles/r01/README.md

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_parity(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}

template <int VER>
struct TmaStage {
    using L = PoolLayout<float, VER>;
    static constexpr int ACT_OFF = L::NVEC * 512 + L::NTAIL * 128;
    static constexpr int BYTES = ACT_OFF + 512;
};

// lane 0 of a warp: request tile `wt` (rows valid envs) into `stage`
template <int VER>
__device__ __forceinline__ void tma_request(const StepParams<float>& p, int64_t wt, unsigned char* stage, uint64_t* bar) {
    using L = PoolLayout<float, VER>;
    const int64_t e0 = wt * 32;
    const int64_t rem = p.n - e0;
    const uint32_t rows = rem < 32 ? (uint32_t)rem : 32u;
    const uint32_t vbytes = rows * 16u;
    const uint32_t b = smem_addr(bar), d = smem_addr(stage);
    mbar_expect_tx(b, (uint32_t)L::TILE_BYTES + vbytes);
    const unsigned char* base = reinterpret_cast<const unsigned char*>(p.pool);
    bulk_g2s(d, base + wt * (int64_t)L::TILE_BYTES, (uint32_t)L::TILE_BYTES, b);     // the whole tile record is one contiguous block
    bulk_g2s(d + TmaStage<VER>::ACT_OFF, p.actions + e0 * 4, vbytes, b);
}

template <int VER, bool MOMENTS>
__global__ void __launch_bounds__(STEP_BLOCK, 4) env_step_tma_kernel(const StepParams<float> p) {
    using Real = float;
    constexpr int OBS = EnvTraits<VER>::OBS;
    constexpr int WARPS = STEP_BLOCK / 32;
    constexpr int SB = TmaStage<VER>::BYTES;
    __shared__ __align__(128) unsigned char s_stage[WARPS][TMA_STAGES][SB];
    __shared__ __align__(8) uint64_t s_bar[WARPS][TMA_STAGES];
    __shared__ float s_tile[WARPS][32 * (OBS + 1)];
    __shared__ double s_mom[MOMENTS ? WARPS : 1][2 * OBS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t warps_total = (int64_t)gridDim.x * WARPS;
    const int64_t n_warp_tiles = (p.n + 31) / 32;
    float* tile = s_tile[warp];
    double m1 = 0.0, m2 = 0.0, G = 0.0;
    if (MOMENTS && lane < OBS) {
        if (p.mom_prev && p.mom_prev[0] > 0.0) G = p.mom_prev[1 + lane];
        else if (p.mom_stats) G = p.mom_stats[1 + lane];
    }
    const int64_t wt0 = (int64_t)blockIdx.x * WARPS + warp;
    if (lane == 0) {
#pragma unroll
        for (int st = 0; st < TMA_STAGES; ++st) mbar_init(smem_addr(&s_bar[warp][st]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int st = 0; st < TMA_STAGES; ++st)
            if (wt0 + st * warps_total < n_warp_tiles) tma_request<VER>(p, wt0 + st * warps_total, s_stage[warp][st], &s_bar[warp][st]);
    }
    __syncwarp();

    int it = 0;
    for (int64_t wt = wt0; wt < n_warp_tiles; wt += warps_total, ++it) {
        const int st = it % TMA_STAGES;
        const uint32_t parity = (uint32_t)(it / TMA_STAGES) & 1u;
        const int64_t e0 = wt * 32;
        const int64_t e = e0 + lane;
        const bool live = e < p.n;
        mbar_wait_parity(smem_addr(&s_bar[warp][st]), parity);
        EnvState<Real, VER> s;
        float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live) {
            pool_load_staged<Real, VER>(s_stage[warp][st], lane, s);
            a4 = *reinterpret_cast<const float4*>(s_stage[warp][st] + TmaStage<VER>::ACT_OFF + lane * 16);
        }
        __syncwarp();                                   // every lane has its tile in registers: the stage can be refilled
        if (lane == 0 && wt + (int64_t)TMA_STAGES * warps_total < n_warp_tiles)
            tma_request<VER>(p, wt + (int64_t)TMA_STAGES * warps_total, s_stage[warp][st], &s_bar[warp][st]);
        float obs[OBS];
        if (live) {
            const float act[4] = {a4.x, a4.y, a4.z, a4.w};
            Real Fcmd, Mcmd[3], F, M[3];
            scale_action<Real>(p.model, act, p.scale_f32, Fcmd, Mcmd);
            mix_and_clamp<Real>(p.model, Fcmd, Mcmd, F, M);
            rk4_step<Real>(p.model, s.y, F, M, p.substeps);
            renormalise_quat<Real>(s.y);
            Real reward;
            int ep_len;
            const uint32_t flags = step_logic<Real, VER>(s, reward, ep_len);
            s.ep_ret += reward;
            make_obs<Real, VER>(s, p.obs_scaled, obs);
            p.reward_out[e] = reward;
            p.flags_out[e] = (uint8_t)flags;
            if (flags & (FLAG_TERMINATED | FLAG_TRUNCATED)) {
                if (p.term_obs_out) {
                    float* row = p.term_obs_out + e * OBS;
#pragma unroll
                    for (int i = 0; i < OBS; ++i) row[i] = obs[i];
                }
                if (p.ep_ret_out) p.ep_ret_out[e] = s.ep_ret;
                if (p.ep_len_out) p.ep_len_out[e] = ep_len;
                if (p.auto_reset) {
                    s.episode += 1;
                    reset_env<Real, VER>(s, p.rc, p.seed, (uint64_t)(p.env_id_offset + e));
                    make_obs<Real, VER>(s, p.obs_scaled, obs);
                }
            }
            pool_store<Real, VER>(p.pool, p.n, e, s);
#pragma unroll
            for (int i = 0; i < OBS; ++i) tile[lane * (OBS + 1) + i] = obs[i];
        }
        __syncwarp();
        const int64_t rem = p.n - e0;
        const int rows = rem < 32 ? (int)rem : 32;
        warp_store_rows<OBS>(p.obs_out + e0 * OBS, tile, lane, rows);
        if (MOMENTS && lane < OBS) {
            const float Lc = tile[lane];
            double t1 = 0.0, t2 = 0.0;
#pragma unroll
            for (int r0 = 0; r0 < 32; r0 += 8) {
                float a1 = 0.f, a2 = 0.f;
#pragma unroll
                for (int r = r0; r < r0 + 8; ++r) {
                    const float v = r < rows ? tile[r * (OBS + 1) + lane] - Lc : 0.f;
                    a1 += v;
                    a2 = fmaf(v, v, a2);
                }
                t1 += (double)a1;
                t2 += (double)a2;
            }
            const double dl = (double)Lc - G;
            m1 += t1 + (double)rows * dl;
            m2 += t2 + 2.0 * dl * t1 + (double)rows * dl * dl;
        }
        __syncwarp();
    }
    if (MOMENTS) {
        if (lane < OBS) { s_mom[warp][lane] = m1; s_mom[warp][OBS + lane] = m2; }
        __syncthreads();
        if (threadIdx.x < 2 * OBS) {
            double a = 0.0;
#pragma unroll
            for (int w = 0; w < WARPS; ++w) a += s_mom[w][threadIdx.x];
            p.mom_partial[(int64_t)blockIdx.x * 2 * OBS + threadIdx.x] = a;
        }
    }
}

// Reset (all envs or a mask) and write their observation; DYN: also draw the new episode's dynamics parameters into `dyn`.
template <typename Real, int VER, bool DYN = false>
__global__ void __launch_bounds__(256) env_reset_kernel(void* pool, int64_t n, const uint8_t* mask, float* obs_out,
                                                         int obs_scaled, uint64_t seed, int64_t env_id_offset,
                                                         ResetConsts rc, int first, Real* dyn, int64_t dyn_stride, DynRand dr) {
    constexpr int OBS = EnvTraits<VER>::OBS;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    if (mask && !mask[e]) return;
    EnvState<Real, VER> s;
    if (first) {
        s.episode = 0;
    } else {
        pool_load<Real, VER>(pool, n, e, s);
        s.episode += 1;
    }
    reset_env<Real, VER>(s, rc, seed, (uint64_t)(env_id_offset + e));
    pool_store<Real, VER>(pool, n, e, s);
    if constexpr (DYN) {
        Real d[N_DYN];
        dyn_redraw(dyn, dyn_stride, dr, (uint64_t)(env_id_offset + e), s.episode, e, d);
    }
    if (obs_out) {
        float obs[OBS];
        make_obs<Real, VER>(s, obs_scaled, obs);
#pragma unroll
        for (int i = 0; i < OBS; ++i) obs_out[e * OBS + i] = obs[i];
    }
}
#endif  // __CUDACC__

}  // namespace qs
