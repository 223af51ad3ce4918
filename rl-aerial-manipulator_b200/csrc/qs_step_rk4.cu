// qs_step_rk4.cu -- instantiations of the fused env-step kernel with the fixed-step RK4 integrator
// (throughput mode), float32 and float64, env v1, v2 and v2 with 2-3 waypoints.
#include "qs_internal.cuh"
#include <stdlib.h>

namespace qs {

template <typename Real, int VER, bool MOMENTS, bool DYN>
static unsigned launch_env_step(qs_handle* h, const StepParams<Real>& p, cudaStream_t st) {
    auto k = env_step_kernel<Real, VER, INTEG_RK4, MOMENTS, DYN>;
    const unsigned grid = step_grid(h, k, STEP_BLOCK);
    k<<<grid, STEP_BLOCK, 0, st>>>(p);
    return grid;
}

template <typename Real>
static int launch_rk4(qs_handle* h, const float* actions, float* obs, Real* reward, uint8_t* flags, float* term_obs,
                      Real* ep_ret, int32_t* ep_len, cudaStream_t st) {
    StepParams<Real> p = base_params<Real>(h);
    p.actions = actions;
    p.obs_out = obs;
    p.reward_out = reward;
    p.flags_out = flags;
    p.term_obs_out = term_obs;
    p.ep_ret_out = ep_ret;
    p.ep_len_out = ep_len;
    p.ls_counters = nullptr;
    p.ls_steps = nullptr;
    unsigned grid = 0;
    QS_FOR_VARIANT(h,
        if (p.dyn) grid = p.mom_partial ? launch_env_step<Real, VER, true, true>(h, p, st) : launch_env_step<Real, VER, false, true>(h, p, st);
        else grid = p.mom_partial ? launch_env_step<Real, VER, true, false>(h, p, st) : launch_env_step<Real, VER, false, false>(h, p, st););
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) {
        set_error(h, "env_step_kernel launch failed: %s", cudaGetErrorString(err));
        return QS_ECUDA;
    }
    if (p.mom_partial) return launch_moments_final(h, grid, st);
    return QS_OK;
}

// float32: QS_STEP_F32_TMA=1 in the environment selects the TMA-fed pipeline kernel (measured slower, see qs_step_kernel.cuh)
template <int VER>
static unsigned launch_tma(qs_handle* h, const StepParams<float>& p, cudaStream_t st) {
    unsigned grid;
    if (p.mom_partial) {
        auto k = env_step_tma_kernel<VER, true>;
        grid = step_grid(h, k, STEP_BLOCK);
        k<<<grid, STEP_BLOCK, 0, st>>>(p);
    } else {
        auto k = env_step_tma_kernel<VER, false>;
        grid = step_grid(h, k, STEP_BLOCK);
        k<<<grid, STEP_BLOCK, 0, st>>>(p);
    }
    return grid;
}

int launch_step_f32(qs_handle* h, const float* actions, float* obs, float* reward, uint8_t* flags, float* term_obs,
                    float* ep_ret, int32_t* ep_len, cudaStream_t st) {
    static const bool use_tma = []() { const char* e = getenv("QS_STEP_F32_TMA"); return e && e[0] == '1'; }();
    if (use_tma && h->dyn_on) {
        set_error(h, "qs_step: the QS_STEP_F32_TMA kernel has no dynamics randomisation; unset QS_STEP_F32_TMA or disarm qs_dynamics_randomization");
        return QS_EINVAL;
    }
    if (!use_tma || (reinterpret_cast<uintptr_t>(actions) & 15)) return launch_rk4<float>(h, actions, obs, reward, flags, term_obs, ep_ret, ep_len, st);
    StepParams<float> p = base_params<float>(h);
    p.actions = actions;
    p.obs_out = obs;
    p.reward_out = reward;
    p.flags_out = flags;
    p.term_obs_out = term_obs;
    p.ep_ret_out = ep_ret;
    p.ep_len_out = ep_len;
    p.ls_counters = nullptr;
    p.ls_steps = nullptr;
    unsigned grid = 0;
    QS_FOR_VARIANT(h, grid = launch_tma<VER>(h, p, st););
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) {
        set_error(h, "env_step_tma_kernel launch failed: %s", cudaGetErrorString(err));
        return QS_ECUDA;
    }
    if (p.mom_partial) return launch_moments_final(h, grid, st);
    return QS_OK;
}

int launch_step_f64(qs_handle* h, const float* actions, float* obs, double* reward, uint8_t* flags, float* term_obs,
                    double* ep_ret, int32_t* ep_len, cudaStream_t st) {
    return launch_rk4<double>(h, actions, obs, reward, flags, term_obs, ep_ret, ep_len, st);
}

}  // namespace qs
