// qs_step_many.cu -- T env steps in ONE launch: the hidden state of an env stays in its thread's registers across the steps.
//
// Why.  At 65,536 envs (BASELINE.json configs[2]) a single step moves 17 MB: the kernel is done in ~3 us and a launch per step
// (even replayed from a CUDA graph) is the floor -- 7.2 us per step measured in r01, 0.37 of the HBM roofline with an L2-resident
// working set.  T steps per launch remove the per-step launch and the per-step state round trip (84 B read + 84 B written per env
// in float32): what is left per env-step is the rollout record, obs 80 B + reward 4 B + flags 1 B (+ 16 B of actions when they
// are read from / written to a buffer).
//
// Same per-env arithmetic as env_step_kernel (the same device functions: scale_action, mix_and_clamp, rk4_step, step_logic,
// make_obs, reset_env), RK4 only, float32 and float64, all three env variants.  Actions come from a time-major buffer
// f32[T, n, 4] or are drawn in the kernel, uniform over the action box: Philox4x32-10 keyed on (action_seed), counter = (global
// env id, step index) -- BASELINE configs[2] "random actions" regenerated on the device every step, shard independent.
// Outputs are time-major [T, n, ...].  A device-resident step counter (advanced by the last CTA to finish) makes consecutive
// launches -- CUDA-graph replays included -- draw fresh actions.
//
// Reference: T iterations of WaypointQuadEnv.step (initial-implementation-v2/rl_env_scaledObs.py:123-231, v1 :85-168) under
// DummyVecEnv.step_wait's auto-reset, for every env of the shard.
#include "qs_internal.cuh"

#include <stdio.h>
#include <string.h>

namespace qs {

template <typename Real>
struct ManyParams {
    StepParams<Real> sp;            // pool, n, model, reset constants (per-call buffers unused)
    int T;
    const float* actions;           // [T, n, 4] or null
    uint64_t action_seed;
    unsigned long long* action_step;   // device counter: first step index of this launch (in-kernel actions)
    float lo[4], span[4];           // action box: a = lo + span * u
    float* actions_out;             // [T, n, 4] or null
    float* obs_out;                 // [T, n, OBS], or [n, OBS] when obs_last_only
    Real* reward_out;               // [T, n]
    uint8_t* flags_out;             // [T, n]
    float* term_obs_out;            // [T, n, OBS] or null
    Real* ep_ret_out;               // [T, n] or null
    int32_t* ep_len_out;            // [T, n] or null
    int obs_last_only;
    unsigned int* ticket;
};

// uniform action of (seed, global env id, step): Philox4x32-10, 24 bits per component
__device__ __forceinline__ float4 philox_uniform_action(uint64_t seed, uint64_t gid, unsigned long long step, const float* lo, const float* span) {
    uint32_t w[4];
    philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)step, (uint32_t)(step >> 32), (uint32_t)seed ^ 0xA4093822u,
                  (uint32_t)(seed >> 32) ^ 0x299F31D0u, w);
    float4 a;
    a.x = fmaf(span[0], (float)(w[0] >> 8) * 5.9604644775390625e-08f, lo[0]);
    a.y = fmaf(span[1], (float)(w[1] >> 8) * 5.9604644775390625e-08f, lo[1]);
    a.z = fmaf(span[2], (float)(w[2] >> 8) * 5.9604644775390625e-08f, lo[2]);
    a.w = fmaf(span[3], (float)(w[3] >> 8) * 5.9604644775390625e-08f, lo[3]);
    return a;
}

// Resident CTAs per SM the kernel is compiled for.  The mode exists for SMALL batches: at 65,536 envs there are 13.8 warps per SM, so
// the float32 kernel is held to 128 registers (4 CTAs = 16 warps per SM: every env resident in one wave, no second round of T
// steps for a leftover third of the warps); float64 needs the registers more (3 CTAs, 168 registers).
template <typename Real> struct ManyOcc { static constexpr int MINB = 3; };
template <> struct ManyOcc<float> { static constexpr int MINB = 4; };

// DYN: dynamics randomisation -- an env's parameters are read once per launch, stay in registers across the T steps, and are
// redrawn (and written back) only where an auto-reset starts a new episode.
template <typename Real, int VER, bool DYN = false>
__global__ void __launch_bounds__(STEP_BLOCK, ManyOcc<Real>::MINB) env_step_many_kernel(const ManyParams<Real> p) {
    constexpr int OBS = EnvTraits<VER>::OBS;
    __shared__ float s_tile[STEP_BLOCK / 32][32 * (OBS + 1)];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const StepParams<Real>& sp = p.sp;
    float* tile = s_tile[warp];
    const int64_t warps_total = (int64_t)gridDim.x * (STEP_BLOCK / 32);
    const int64_t n_warp_tiles = (sp.n + 31) / 32;
    unsigned long long step0 = 0;
    if (!p.actions && p.action_step) step0 = *reinterpret_cast<const volatile unsigned long long*>(p.action_step);

    for (int64_t wt = (int64_t)blockIdx.x * (STEP_BLOCK / 32) + warp; wt < n_warp_tiles; wt += warps_total) {
        const int64_t e0 = wt * 32, e = e0 + lane;
        const bool live = e < sp.n;
        const int64_t rem = sp.n - e0;
        const int rows = rem < 32 ? (int)rem : 32;
        EnvState<Real, VER> s;
        if (live) pool_load<Real, VER>(sp.pool, sp.n, e, s);
        Real d[DYN ? N_DYN : 1];
        if constexpr (DYN) {
            if (live) dyn_load(sp, e, d);
        }
        float4 a_next = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live && p.actions) a_next = __ldcs(reinterpret_cast<const float4*>(p.actions) + e);
#pragma unroll 1
        for (int t = 0; t < p.T; ++t) {
            const int64_t row = (int64_t)t * sp.n + e;
            float obs[OBS];
            if (live) {
                float4 a4;
                if (p.actions) {
                    a4 = a_next;                                        // the next step's action is in flight while this one integrates
                    if (t + 1 < p.T) a_next = __ldcs(reinterpret_cast<const float4*>(p.actions) + row + sp.n);
                } else {
                    a4 = philox_uniform_action(p.action_seed, (uint64_t)(sp.env_id_offset + e), step0 + (unsigned long long)t, p.lo, p.span);
                }
                if (p.actions_out) __stcs(reinterpret_cast<float4*>(p.actions_out) + row, a4);
                const float act[4] = {a4.x, a4.y, a4.z, a4.w};
                Real Fcmd, Mcmd[3], F, M[3];
                scale_action<Real>(sp.model, act, sp.scale_f32, Fcmd, Mcmd);
                if constexpr (DYN) {
                    Real aw[3];
                    dyn_forces<Real>(sp.model, Fcmd, Mcmd, d, F, M, aw);
                    rk4_step<Real, true>(sp.model, s.y, F, M, sp.substeps, aw);
                } else {
                    mix_and_clamp<Real>(sp.model, Fcmd, Mcmd, F, M);
                    rk4_step<Real>(sp.model, s.y, F, M, sp.substeps);
                }
                renormalise_quat<Real>(s.y);
                Real reward;
                int ep_len;
                const uint32_t flags = step_logic<Real, VER>(s, reward, ep_len);
                s.ep_ret += reward;
                make_obs<Real, VER>(s, sp.obs_scaled, obs);
                __stcs(p.reward_out + row, reward);
                p.flags_out[row] = (uint8_t)flags;
                if (flags & (FLAG_TERMINATED | FLAG_TRUNCATED)) {
                    if (p.term_obs_out) {
                        float* trow = p.term_obs_out + row * OBS;
#pragma unroll
                        for (int i = 0; i < OBS; ++i) trow[i] = obs[i];
                    }
                    if (p.ep_ret_out) p.ep_ret_out[row] = s.ep_ret;
                    if (p.ep_len_out) p.ep_len_out[row] = ep_len;
                    if (sp.auto_reset) {
                        s.episode += 1;
                        reset_env<Real, VER>(s, sp.rc, sp.seed, (uint64_t)(sp.env_id_offset + e));
                        make_obs<Real, VER>(s, sp.obs_scaled, obs);
                        if constexpr (DYN) dyn_redraw(sp.dyn, sp.dyn_stride, sp.dr, (uint64_t)(sp.env_id_offset + e), s.episode, e, d);
                    }
                }
            }
            if (!p.obs_last_only || t == p.T - 1) {
                if (live) {
#pragma unroll
                    for (int i = 0; i < OBS; ++i) tile[lane * (OBS + 1) + i] = obs[i];
                }
                __syncwarp();
                float* dst = p.obs_last_only ? p.obs_out + e0 * OBS : p.obs_out + ((int64_t)t * sp.n + e0) * OBS;
                warp_store_rows<OBS>(dst, tile, lane, rows);
                __syncwarp();
            }
        }
        if (live) pool_store<Real, VER>(sp.pool, sp.n, e, s);
    }
    // the last CTA to finish advances the action step counter (every CTA has read it by then)
    if (!p.actions && p.action_step) {
        __shared__ unsigned int s_last;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = atomicAdd(p.ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
        __syncthreads();
        if (s_last && threadIdx.x == 0) {
            *p.ticket = 0u;
            *p.action_step = step0 + (unsigned long long)p.T;
        }
    }
}

template <typename Real>
static int launch_many(qs_handle* h, const qs_step_many_args* a, cudaStream_t st) {
    ManyParams<Real> p;
    memset(&p, 0, sizeof(p));
    p.sp = base_params<Real>(h);
    p.T = a->T;
    p.actions = a->actions;
    p.action_seed = a->action_seed;
    p.action_step = reinterpret_cast<unsigned long long*>(a->action_step);
    for (int i = 0; i < 4; ++i) { p.lo[i] = a->action_lo[i]; p.span[i] = a->action_hi[i] - a->action_lo[i]; }
    p.actions_out = a->actions_out;
    p.obs_out = a->obs_out;
    p.reward_out = static_cast<Real*>(a->reward_out);
    p.flags_out = a->flags_out;
    p.term_obs_out = a->terminal_obs_out;
    p.ep_ret_out = static_cast<Real*>(a->ep_return_out);
    p.ep_len_out = a->ep_len_out;
    p.obs_last_only = a->obs_last_only;
    p.ticket = h->ro_ticket;
    cudaError_t err = cudaSuccess;
    QS_FOR_VARIANT(h, {
        auto k = p.sp.dyn ? env_step_many_kernel<Real, VER, true> : env_step_many_kernel<Real, VER, false>;
        const unsigned grid = step_grid(h, k, STEP_BLOCK);
        k<<<grid, STEP_BLOCK, 0, st>>>(p);
    });
    err = cudaGetLastError();
    if (err != cudaSuccess) { set_error(h, "env_step_many_kernel launch failed: %s", cudaGetErrorString(err)); return QS_ECUDA; }
    return QS_OK;
}

}  // namespace qs

using namespace qs;

extern "C" int qs_step_many(qs_handle* h, const qs_step_many_args* a, void* stream) {
    if (!h || !a) { set_error(h, "qs_step_many: null argument"); return QS_EINVAL; }
    if (h->cfg.integrator != QS_RK4) { set_error(h, "qs_step_many: RK4 handles only"); return QS_EINVAL; }
    if (!h->initialized) { set_error(h, "qs_step_many: call qs_reset first"); return QS_EINVAL; }
    if (h->mom_out) { set_error(h, "qs_step_many: not available while qs_step_moments is armed"); return QS_EINVAL; }
    if (a->T < 1 || !a->obs_out || !a->reward_out || !a->flags_out) { set_error(h, "qs_step_many: T >= 1, obs_out, reward_out and flags_out are required"); return QS_EINVAL; }
    if (!a->actions && !a->action_step) { set_error(h, "qs_step_many: pass actions f32[T,n,4] or a device step counter for in-kernel actions"); return QS_EINVAL; }
    if ((reinterpret_cast<uintptr_t>(a->actions) | reinterpret_cast<uintptr_t>(a->actions_out) | reinterpret_cast<uintptr_t>(a->obs_out)) & 15) {
        set_error(h, "qs_step_many: actions, actions_out and obs_out must be 16-byte aligned");
        return QS_EINVAL;
    }
    if (!a->obs_last_only && (((int64_t)h->cfg.n_envs * (h->cfg.env_version == 2 ? 20 : 17)) & 3)) {
        set_error(h, "qs_step_many: n_envs * obs_dim must be a multiple of 4 for time-major obs (128-bit row stores); use obs_last_only");
        return QS_EINVAL;
    }
    cudaError_t err = cudaSetDevice(h->cfg.device);
    if (err != cudaSuccess) { set_error(h, "qs_step_many: cudaSetDevice: %s", cudaGetErrorString(err)); return QS_ECUDA; }
    if (!h->ro_ticket) {
        err = cudaMalloc(&h->ro_ticket, sizeof(unsigned int));
        if (err == cudaSuccess) err = cudaMemset(h->ro_ticket, 0, sizeof(unsigned int));
        if (err != cudaSuccess) { set_error(h, "qs_step_many: ticket allocation: %s", cudaGetErrorString(err)); return QS_ECUDA; }
    }
    return h->cfg.precision == QS_F32 ? launch_many<float>(h, a, (cudaStream_t)stream) : launch_many<double>(h, a, (cudaStream_t)stream);
}
