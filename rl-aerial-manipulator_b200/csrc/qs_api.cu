// qs_api.cu -- C ABI of libquadsim.so (include/quadsim.h): handle lifecycle, dispatch to the sm_100a kernels,
// state injection/extraction.  No torch types, no C++ exceptions across the boundary.
#include "../../include/quadsim.h"
#include "qs_internal.cuh"
#include "qs_exchange.cuh"

#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <new>

namespace qs {
thread_local char g_error[512] = "";

void set_error(qs_handle* h, const char* fmt, ...) {
    char* dst = h ? h->error : g_error;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(dst, 512, fmt, ap);
    va_end(ap);
}

// ---- canonical f64 view <-> pool ---------------------------------------------------------------------
template <typename Real, int VER>
__global__ void get_state_kernel(const void* pool, int64_t n, qs_state_view v) {
    constexpr int NWP = EnvTraits<VER>::NWP;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    EnvState<Real, VER> s;
    pool_load<Real, VER>(pool, n, e, s);
    if (v.y) for (int i = 0; i < 13; ++i) v.y[e * 13 + i] = (double)s.y[i];
    if (v.wp_list)
        for (int j = 0; j < QS_MAX_WAYPOINTS; ++j)
            for (int i = 0; i < 3; ++i) v.wp_list[(e * QS_MAX_WAYPOINTS + j) * 3 + i] = j < NWP ? (double)s.wp[j][i] : 0.0;
    if (v.n_wp) v.n_wp[e] = s.n_wp();
    if (v.wp_index) v.wp_index[e] = s.wp_index();
    if (v.last_distance) v.last_distance[e] = s.has_last() ? (double)s.last_d : nan("");
    if (v.current_step) v.current_step[e] = s.step();
    if (v.counter) v.counter[e] = s.counter();
    if (v.final_reached) v.final_reached[e] = s.final_reached() ? 1 : 0;
    if (v.final_yaw) v.final_yaw[e] = (double)s.final_yaw;
    if (v.ep_return) v.ep_return[e] = (double)s.ep_ret;
    if (v.episode) v.episode[e] = (int32_t)s.episode;
}

template <typename Real, int VER>
__global__ void set_state_kernel(void* pool, int64_t n, qs_state_view v) {
    constexpr int NWP = EnvTraits<VER>::NWP;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    EnvState<Real, VER> s;
    pool_load<Real, VER>(pool, n, e, s);
    if (v.y) for (int i = 0; i < 13; ++i) s.y[i] = (Real)v.y[e * 13 + i];
    if (v.wp_list)
        for (int j = 0; j < NWP; ++j)
            for (int i = 0; i < 3; ++i) s.wp[j][i] = (Real)v.wp_list[(e * QS_MAX_WAYPOINTS + j) * 3 + i];
    int step = s.step(), counter = s.counter(), idx = s.wp_index(), nwp = s.n_wp();
    bool fin = s.final_reached(), has_last = s.has_last();
    if (v.n_wp) nwp = v.n_wp[e];
    if (v.wp_index) idx = v.wp_index[e];
    if (v.last_distance) {
        const double d = v.last_distance[e];
        has_last = !isnan(d);
        s.last_d = has_last ? (Real)d : Real(0);
    }
    if (v.current_step) step = v.current_step[e];
    if (v.counter) counter = v.counter[e];
    if (v.final_reached) fin = v.final_reached[e] != 0;
    if (v.final_yaw) s.final_yaw = (Real)v.final_yaw[e];
    if (v.ep_return) s.ep_ret = (Real)v.ep_return[e];
    if (v.episode) s.episode = (uint32_t)v.episode[e];
    s.set(step, counter, idx, nwp, fin, has_last);
    pool_store<Real, VER>(pool, n, e, s);
}

__global__ void reset_uniforms_kernel(uint64_t seed, const int64_t* env_ids, const int32_t* episodes, int64_t n, double* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double u[QS_N_UNIFORMS];
    reset_uniforms(seed, (uint64_t)env_ids[i], (uint32_t)episodes[i], u);
    for (int k = 0; k < QS_N_UNIFORMS; ++k) out[i * QS_N_UNIFORMS + k] = u[k];
}

// ---- dynamics randomisation planes <-> f64 rows -------------------------------------------------------------
// arming a reset handle: every env's parameters for the episode it is in
template <typename Real, int VER>
__global__ void dyn_arm_kernel(const void* pool, int64_t n, Real* dyn, int64_t stride, DynRand dr, int64_t env_id_offset) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    EnvState<Real, VER> s;
    pool_load<Real, VER>(pool, n, e, s);
    Real d[N_DYN];
    dyn_redraw(dyn, stride, dr, (uint64_t)(env_id_offset + e), s.episode, e, d);
}

template <typename Real>
__global__ void dyn_get_kernel(const Real* dyn, int64_t stride, int64_t n, double* out) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    for (int k = 0; k < N_DYN; ++k) out[e * N_DYN + k] = (double)dyn[k * stride + e];
}

template <typename Real>
__global__ void dyn_set_kernel(Real* dyn, int64_t stride, int64_t n, const double* in) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    for (int k = 0; k < N_DYN; ++k) dyn[k * stride + e] = (Real)in[e * N_DYN + k];
}

template <typename Real, int VER>
static size_t pool_bytes(int64_t n) { return (size_t)PoolLayout<Real, VER>::TILE_BYTES * (size_t)((n + 31) / 32); }   // whole warp tiles

static bool near_zero(double v) { return fabs(v) < 1e-300; }

}  // namespace qs

using namespace qs;

#define QS_CUDA(h, call)                                                                     \
    do {                                                                                     \
        cudaError_t err__ = (call);                                                          \
        if (err__ != cudaSuccess) {                                                          \
            set_error(h, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), __FILE__, __LINE__); \
            return QS_ECUDA;                                                                 \
        }                                                                                    \
    } while (0)

// dispatch on (precision, env_version): BODY sees `Real` and `VER`
#define QS_DISPATCH(h, ...)                                     \
    do {                                                        \
        if ((h)->cfg.precision == QS_F32) {                     \
            using Real = float;                                 \
            QS_FOR_VARIANT(h, __VA_ARGS__);                     \
        } else {                                                \
            using Real = double;                                \
            QS_FOR_VARIANT(h, __VA_ARGS__);                     \
        }                                                       \
    } while (0)

extern "C" {

int qs_abi_version(void) { return QS_ABI_VERSION; }

const char* qs_last_error(const qs_handle* h) { return h ? h->error : g_error; }

int qs_create(const qs_config* cfg, qs_handle** out) {
    if (!cfg || !out) { set_error(nullptr, "qs_create: null argument"); return QS_EINVAL; }
    *out = nullptr;
    if (cfg->abi_version != QS_ABI_VERSION) { set_error(nullptr, "qs_create: abi_version %d != %d", cfg->abi_version, QS_ABI_VERSION); return QS_EINVAL; }
    if (cfg->env_version != 1 && cfg->env_version != 2) { set_error(nullptr, "qs_create: env_version must be 1 or 2"); return QS_EINVAL; }
    if (cfg->precision != QS_F32 && cfg->precision != QS_F64) { set_error(nullptr, "qs_create: bad precision"); return QS_EINVAL; }
    if (cfg->integrator != QS_RK4 && cfg->integrator != QS_LSODA) { set_error(nullptr, "qs_create: bad integrator"); return QS_EINVAL; }
    if (cfg->integrator == QS_LSODA && cfg->precision != QS_F64) { set_error(nullptr, "qs_create: QS_LSODA requires QS_F64"); return QS_EINVAL; }
    if (cfg->integrator == QS_RK4 && cfg->substeps < 1) { set_error(nullptr, "qs_create: substeps must be >= 1"); return QS_EINVAL; }
    if (cfg->n_envs < 1) { set_error(nullptr, "qs_create: n_envs must be >= 1"); return QS_EINVAL; }
    if (cfg->v2_random_waypoints && cfg->env_version != 2) { set_error(nullptr, "qs_create: v2_random_waypoints needs env_version 2"); return QS_EINVAL; }
    if (cfg->env_version == 2 && !cfg->obs_scaled) { set_error(nullptr, "qs_create: v2 has no raw-observation variant"); return QS_EINVAL; }
    const int zero_idx[4] = {1, 3, 5, 7};
    for (int k = 0; k < 4; ++k)
        if (!near_zero(cfg->inertia[zero_idx[k]]) || !near_zero(cfg->inv_inertia[zero_idx[k]])) {
            set_error(nullptr, "qs_create: inertia must have zeros at (0,1),(1,0),(1,2),(2,1) like the reference's");
            return QS_EINVAL;
        }
    if (!(cfg->mass > 0) || !(cfg->dt > 0)) { set_error(nullptr, "qs_create: mass and dt must be positive"); return QS_EINVAL; }

    int ndev = 0;
    cudaError_t err = cudaGetDeviceCount(&ndev);
    if (err != cudaSuccess || ndev == 0) {
        set_error(nullptr, "qs_create: no CUDA device (%s); libquadsim has no CPU fallback", cudaGetErrorString(err));
        return QS_ECUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) { set_error(nullptr, "qs_create: device %d out of range (%d devices)", cfg->device, ndev); return QS_EINVAL; }
    QS_CUDA(nullptr, cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    QS_CUDA(nullptr, cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) {
        set_error(nullptr, "qs_create: device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);
        return QS_EINVAL;
    }

    qs_handle* h = new (std::nothrow) qs_handle();
    if (!h) { set_error(nullptr, "qs_create: out of host memory"); return QS_ENOMEM; }
    h->cfg = *cfg;
    h->error[0] = 0;
    h->num_sms = prop.multiProcessorCount;
    h->initialized = false;
    size_t bytes = 0;
    QS_DISPATCH(h, bytes = pool_bytes<Real, VER>(cfg->n_envs); h->bytes_per_env = PoolLayout<Real, VER>::BYTES;);
    h->pool_bytes = bytes;
    err = cudaMalloc(&h->pool, bytes + 4096);
    if (err != cudaSuccess) {
        set_error(nullptr, "qs_create: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(err));
        delete h;
        return QS_ENOMEM;
    }
    cudaMemset(h->pool, 0, bytes + 4096);
    h->mom_scratch = nullptr;
    h->mom_out = nullptr;
    h->mom_stats = nullptr;
    h->mom_merge = nullptr;
    h->mom_xchg = nullptr;
    h->mom_xchg_stats = nullptr;
    h->range_first = 0;
    h->range_count = 0;
    // last-CTA election counter of qs_rollout_step / qs_step_many: allocated here, not lazily, so that the first call of either may
    // already be inside a CUDA-graph capture (cudaMemset on the legacy stream is illegal there)
    h->ro_ticket = nullptr;
    if (cudaMalloc(&h->ro_ticket, sizeof(unsigned int)) != cudaSuccess || cudaMemset(h->ro_ticket, 0, sizeof(unsigned int)) != cudaSuccess) {
        set_error(nullptr, "qs_create: ticket allocation failed");
        cudaFree(h->pool);
        delete h;
        return QS_ENOMEM;
    }
    h->ls_tables = nullptr;
    h->ls_counters = nullptr;
    h->ls_steps = nullptr;
    if (cfg->integrator == QS_LSODA) {
        LsodaTables T;
        lsoda_tables_init(T);
        err = cudaMalloc(&h->ls_tables, sizeof(T));
        if (err == cudaSuccess) err = cudaMemcpy(h->ls_tables, &T, sizeof(T), cudaMemcpyHostToDevice);
        if (err == cudaSuccess) err = cudaMalloc(&h->ls_counters, sizeof(int32_t) * 4 * cfg->n_envs);
        if (err == cudaSuccess) err = cudaMalloc(&h->ls_steps, sizeof(double) * 2 * cfg->n_envs);
        if (err != cudaSuccess) {
            set_error(nullptr, "qs_create: LSODA setup failed: %s", cudaGetErrorString(err));
            qs_destroy(h);
            return QS_ECUDA;
        }
    }
    *out = h;
    return QS_OK;
}

int qs_destroy(qs_handle* h) {
    if (!h) return QS_OK;
    cudaSetDevice(h->cfg.device);
    if (h->pool) cudaFree(h->pool);
    if (h->mom_scratch) cudaFree(h->mom_scratch);
    if (h->ro_ticket) cudaFree(h->ro_ticket);
    if (h->ls_tables) cudaFree(h->ls_tables);
    if (h->ls_counters) cudaFree(h->ls_counters);
    if (h->ls_steps) cudaFree(h->ls_steps);
    if (h->dyn) cudaFree(h->dyn);
    delete h;
    return QS_OK;
}

int qs_obs_dim(const qs_handle* h) { return h ? (h->cfg.env_version == 2 ? 20 : 17) : QS_EINVAL; }

int64_t qs_state_bytes_per_env(const qs_handle* h) { return h ? h->bytes_per_env : QS_EINVAL; }

int qs_reset(qs_handle* h, const uint8_t* env_mask, float* obs_out, void* stream) {
    if (!h) { set_error(nullptr, "qs_reset: null handle"); return QS_EINVAL; }
    if (env_mask && !h->initialized) { set_error(h, "qs_reset: the first reset must cover all envs (env_mask == NULL)"); return QS_EINVAL; }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = h->cfg.n_envs;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    ResetConsts rc;
    for (int i = 0; i < QS_TRIG_TAB; ++i) { rc.sin_tab[i] = h->cfg.sin_tab[i]; rc.cos_tab[i] = h->cfg.cos_tab[i]; }
    QS_DISPATCH(h, {
        Real* dyn = static_cast<Real*>(h->dyn);
        auto k = h->dyn_on ? env_reset_kernel<Real, VER, true> : env_reset_kernel<Real, VER, false>;
        k<<<blocks, 256, 0, st>>>(h->pool, n, env_mask, obs_out, h->cfg.obs_scaled, h->cfg.seed, h->cfg.env_id_offset, rc,
                                  h->initialized ? 0 : 1, dyn, h->dyn_stride, h->dyn_cfg);
    });
    QS_CUDA(h, cudaGetLastError());
    h->initialized = true;
    return QS_OK;
}

int qs_step(qs_handle* h, const float* actions, float* obs_out, void* reward_out, uint8_t* flags_out,
            float* terminal_obs_out, void* ep_return_out, int32_t* ep_len_out, void* stream) {
    if (!h) { set_error(nullptr, "qs_step: null handle"); return QS_EINVAL; }
    if (!actions || !obs_out || !reward_out || !flags_out) { set_error(h, "qs_step: actions, obs_out, reward_out and flags_out are required"); return QS_EINVAL; }
    if (!h->initialized) { set_error(h, "qs_step: call qs_reset first"); return QS_EINVAL; }
    // the kernels read an action row with one LDG.128 and write obs rows with STG.128: a misaligned pointer would be a sticky
    // misaligned-address fault instead of an error code
    if ((reinterpret_cast<uintptr_t>(actions) | reinterpret_cast<uintptr_t>(obs_out)) & 15) {
        set_error(h, "qs_step: actions and obs_out must be 16-byte aligned");
        return QS_EINVAL;
    }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    int rc = QS_OK;
    if (h->cfg.precision == QS_F32)
        rc = launch_step_f32(h, actions, obs_out, (float*)reward_out, flags_out, terminal_obs_out, (float*)ep_return_out, ep_len_out, (cudaStream_t)stream);
    else if (h->cfg.integrator == QS_RK4)
        rc = launch_step_f64(h, actions, obs_out, (double*)reward_out, flags_out, terminal_obs_out, (double*)ep_return_out, ep_len_out, (cudaStream_t)stream);
    else
        rc = launch_step_lsoda(h, actions, obs_out, (double*)reward_out, flags_out, terminal_obs_out, (double*)ep_return_out, ep_len_out, (cudaStream_t)stream);
    return rc;
}

int qs_step_range(qs_handle* h, int64_t first_env, int64_t count, const float* actions, float* obs_out, void* reward_out,
                  uint8_t* flags_out, float* terminal_obs_out, void* ep_return_out, int32_t* ep_len_out, void* stream) {
    if (!h) { set_error(nullptr, "qs_step_range: null handle"); return QS_EINVAL; }
    if (first_env < 0 || count < 1 || (first_env & 31) || first_env + count > h->cfg.n_envs) {
        set_error(h, "qs_step_range: need 0 <= first_env (multiple of 32), count >= 1, first_env + count <= n_envs");
        return QS_EINVAL;
    }
    if (h->cfg.integrator != QS_RK4) { set_error(h, "qs_step_range: RK4 handles only"); return QS_EINVAL; }
    if (h->mom_out) { set_error(h, "qs_step_range: not available while qs_step_moments is armed"); return QS_EINVAL; }
    h->range_first = first_env;
    h->range_count = count;
    const int rc = qs_step(h, actions, obs_out, reward_out, flags_out, terminal_obs_out, ep_return_out, ep_len_out, stream);
    h->range_first = 0;
    h->range_count = 0;
    return rc;
}

int qs_step_moments(qs_handle* h, double* moments_out, const double* shift_stats) {
    if (!h) { set_error(nullptr, "qs_step_moments: null handle"); return QS_EINVAL; }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    if (moments_out && !h->mom_scratch) {
        const int d = h->cfg.env_version == 2 ? 20 : 17;
        // upper bound of any step grid: 16 resident CTAs of 128 threads per SM
        QS_CUDA(h, cudaMalloc(&h->mom_scratch, sizeof(double) * 2 * d * (size_t)h->num_sms * 16));
    }
    h->mom_out = moments_out;
    h->mom_stats = moments_out ? shift_stats : nullptr;
    if (!moments_out) { h->mom_merge = nullptr; h->mom_xchg = nullptr; h->mom_xchg_stats = nullptr; }
    return QS_OK;
}

int qs_step_moments_exchange(qs_handle* h, qs_xchg* x, double* stats) {
    if (!h) { set_error(nullptr, "qs_step_moments_exchange: null handle"); return QS_EINVAL; }
    if (!x) { h->mom_xchg = nullptr; h->mom_xchg_stats = nullptr; return QS_OK; }
    if (!h->mom_out) { set_error(h, "qs_step_moments_exchange: arm qs_step_moments first"); return QS_EINVAL; }
    if (!stats) { set_error(h, "qs_step_moments_exchange: null statistics"); return QS_EINVAL; }
    if (h->mom_merge) { set_error(h, "qs_step_moments_exchange: qs_step_moments_merge is armed (the exchange does the merge)"); return QS_EINVAL; }
    const int d = h->cfg.env_version == 2 ? 20 : 17;
    if (x->d != d || !x->connected) {
        set_error(h, "qs_step_moments_exchange: the exchange must be connected and have the env's observation width (%d)", d);
        return QS_EINVAL;
    }
    h->mom_xchg = x;
    h->mom_xchg_stats = stats;
    return QS_OK;
}

int qs_step_moments_merge(qs_handle* h, double* merge_stats) {
    if (!h) { set_error(nullptr, "qs_step_moments_merge: null handle"); return QS_EINVAL; }
    if (merge_stats && !h->mom_out) { set_error(h, "qs_step_moments_merge: arm qs_step_moments first"); return QS_EINVAL; }
    if (merge_stats && h->mom_xchg) { set_error(h, "qs_step_moments_merge: qs_step_moments_exchange is armed (the exchange does the merge)"); return QS_EINVAL; }
    h->mom_merge = merge_stats;
    return QS_OK;
}

int qs_get_state(qs_handle* h, const qs_state_view* out, void* stream) {
    if (!h || !out) { set_error(h, "qs_get_state: null argument"); return QS_EINVAL; }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    const int64_t n = h->cfg.n_envs;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    QS_DISPATCH(h, (get_state_kernel<Real, VER><<<blocks, 128, 0, (cudaStream_t)stream>>>(h->pool, n, *out)););
    QS_CUDA(h, cudaGetLastError());
    return QS_OK;
}

int qs_set_state(qs_handle* h, const qs_state_view* in, void* stream) {
    if (!h || !in) { set_error(h, "qs_set_state: null argument"); return QS_EINVAL; }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    const int64_t n = h->cfg.n_envs;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    QS_DISPATCH(h, (set_state_kernel<Real, VER><<<blocks, 128, 0, (cudaStream_t)stream>>>(h->pool, n, *in)););
    QS_CUDA(h, cudaGetLastError());
    h->initialized = true;
    return QS_OK;
}

int qs_reset_uniforms(qs_handle* h, const int64_t* env_ids, const int32_t* episodes, int64_t n, double* out, void* stream) {
    if (!h || !env_ids || !episodes || !out || n < 0) { set_error(h, "qs_reset_uniforms: bad argument"); return QS_EINVAL; }
    if (n == 0) return QS_OK;
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    reset_uniforms_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(h->cfg.seed, env_ids, episodes, n, out);
    QS_CUDA(h, cudaGetLastError());
    return QS_OK;
}

int qs_dynamics_randomization(qs_handle* h, const qs_dynamics_rand* cfg, void* stream) {
    if (!h) { set_error(nullptr, "qs_dynamics_randomization: null handle"); return QS_EINVAL; }
    if (!cfg) { h->dyn_on = false; return QS_OK; }
    if (h->cfg.integrator != QS_RK4) { set_error(h, "qs_dynamics_randomization: RK4 handles only (no dynamics randomisation in QS_LSODA)"); return QS_EINVAL; }
    const bool ok = isfinite(cfg->mass_rel) && isfinite(cfg->inertia_rel) && isfinite(cfg->thrust_rel) && isfinite(cfg->wind) &&
                    cfg->mass_rel >= 0 && cfg->mass_rel < 1 && cfg->inertia_rel >= 0 && cfg->inertia_rel < 1 &&
                    cfg->thrust_rel >= 0 && cfg->thrust_rel <= 1 && cfg->wind >= 0;
    if (!ok) {
        set_error(h, "qs_dynamics_randomization: need finite 0 <= mass_rel < 1, 0 <= inertia_rel < 1, 0 <= thrust_rel <= 1, wind >= 0");
        return QS_EINVAL;
    }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    const int64_t n = h->cfg.n_envs;
    if (!h->dyn) {
        h->dyn_stride = (n + 31) / 32 * 32;
        const size_t real = h->cfg.precision == QS_F32 ? sizeof(float) : sizeof(double);
        QS_CUDA(h, cudaMalloc(&h->dyn, real * QS_DYN_PARAMS * (size_t)h->dyn_stride));
    }
    h->dyn_cfg.seed = cfg->seed;
    h->dyn_cfg.mass_rel = cfg->mass_rel;
    h->dyn_cfg.inertia_rel = cfg->inertia_rel;
    h->dyn_cfg.thrust_rel = cfg->thrust_rel;
    h->dyn_cfg.wind = cfg->wind;
    h->dyn_on = true;
    // every env's parameters for the episode its record holds (0 in the zeroed pool of a handle that was never reset)
    const unsigned blocks = (unsigned)((n + 127) / 128);
    QS_DISPATCH(h, (dyn_arm_kernel<Real, VER><<<blocks, 128, 0, (cudaStream_t)stream>>>(h->pool, n, static_cast<Real*>(h->dyn), h->dyn_stride,
                                                                                    h->dyn_cfg, h->cfg.env_id_offset)););
    QS_CUDA(h, cudaGetLastError());
    return QS_OK;
}

int qs_get_dynamics(qs_handle* h, double* out, void* stream) {
    if (!h || !out) { set_error(h, "qs_get_dynamics: null argument"); return QS_EINVAL; }
    if (!h->dyn_on) { set_error(h, "qs_get_dynamics: dynamics randomisation is not armed (qs_dynamics_randomization)"); return QS_EINVAL; }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    const int64_t n = h->cfg.n_envs;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    if (h->cfg.precision == QS_F32) dyn_get_kernel<float><<<blocks, 128, 0, (cudaStream_t)stream>>>(static_cast<float*>(h->dyn), h->dyn_stride, n, out);
    else dyn_get_kernel<double><<<blocks, 128, 0, (cudaStream_t)stream>>>(static_cast<double*>(h->dyn), h->dyn_stride, n, out);
    QS_CUDA(h, cudaGetLastError());
    return QS_OK;
}

int qs_set_dynamics(qs_handle* h, const double* in, void* stream) {
    if (!h || !in) { set_error(h, "qs_set_dynamics: null argument"); return QS_EINVAL; }
    if (!h->dyn_on) { set_error(h, "qs_set_dynamics: dynamics randomisation is not armed (qs_dynamics_randomization)"); return QS_EINVAL; }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    const int64_t n = h->cfg.n_envs;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    if (h->cfg.precision == QS_F32) dyn_set_kernel<float><<<blocks, 128, 0, (cudaStream_t)stream>>>(static_cast<float*>(h->dyn), h->dyn_stride, n, in);
    else dyn_set_kernel<double><<<blocks, 128, 0, (cudaStream_t)stream>>>(static_cast<double*>(h->dyn), h->dyn_stride, n, in);
    QS_CUDA(h, cudaGetLastError());
    return QS_OK;
}

int qs_lsoda_stats(qs_handle* h, int32_t* counters_out, double* steps_out, void* stream) {
    if (!h) { set_error(nullptr, "qs_lsoda_stats: null handle"); return QS_EINVAL; }
    if (h->cfg.integrator != QS_LSODA) { set_error(h, "qs_lsoda_stats: handle is not in QS_LSODA mode"); return QS_EINVAL; }
    QS_CUDA(h, cudaSetDevice(h->cfg.device));
    const int64_t n = h->cfg.n_envs;
    if (counters_out) QS_CUDA(h, cudaMemcpyAsync(counters_out, h->ls_counters, sizeof(int32_t) * 4 * n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    if (steps_out) QS_CUDA(h, cudaMemcpyAsync(steps_out, h->ls_steps, sizeof(double) * 2 * n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return QS_OK;
}

}  // extern "C"
