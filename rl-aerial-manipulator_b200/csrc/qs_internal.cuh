// qs_internal.cuh -- handle definition and launcher prototypes shared by the translation units of libquadsim.
#pragma once
#include "../../include/quadsim.h"
#include "qs_step_kernel.cuh"
#include <cuda_runtime.h>

struct qs_handle {
    qs_config cfg;
    void* pool;
    size_t pool_bytes;
    int64_t bytes_per_env;
    double* mom_scratch;      // fused obs moments: per-CTA partials [grid][2*obs_dim]; null = off
    double* mom_out;          // caller-owned (n, mean[D], M2[D]) triplet
    const double* mom_stats;  // caller-owned VecNormalize stats used as the shift (or null)
    double* mom_merge;        // caller-owned running statistics the batch triplet is merged into by the step (or null)
    struct qs_xchg* mom_xchg; // several ranks: the peer-memory exchange the kernel that finishes the moments also runs (or null)
    double* mom_xchg_stats;   // ... and the running statistics the exchanged triplets are merged into
    qs::LsodaTables* ls_tables;
    int32_t* ls_counters;
    double* ls_steps;
    unsigned int* ro_ticket;  // qs_rollout_step: last-CTA election counter
    int64_t range_first, range_count;   // qs_step_range: the sub-range the next launch covers (count 0 = all envs)
    void* dyn;                // dynamics randomisation: Real planes [QS_DYN_PARAMS][dyn_stride]; null = never armed
    int64_t dyn_stride;       // n_envs rounded up to whole warp tiles
    bool dyn_on;              // armed (qs_dynamics_randomization)
    qs::DynRand dyn_cfg;
    int num_sms;
    bool initialized;
    char error[512];
};

namespace qs {
void set_error(qs_handle* h, const char* fmt, ...);

// (n, mean, M2) from the per-CTA partials a step kernel launched with `blocks` CTAs left in h->mom_scratch (qs_vecnorm.cu)
int launch_moments_final(qs_handle* h, unsigned blocks, cudaStream_t st);

int launch_step_f32(qs_handle* h, const float* actions, float* obs, float* reward, uint8_t* flags, float* term_obs,
                    float* ep_ret, int32_t* ep_len, cudaStream_t st);
int launch_step_f64(qs_handle* h, const float* actions, float* obs, double* reward, uint8_t* flags, float* term_obs,
                    double* ep_ret, int32_t* ep_len, cudaStream_t st);
int launch_step_lsoda(qs_handle* h, const float* actions, float* obs, double* reward, uint8_t* flags, float* term_obs,
                      double* ep_ret, int32_t* ep_len, cudaStream_t st);

// Fill StepParams from the handle (everything except the per-call buffers).
template <typename Real>
inline StepParams<Real> base_params(const qs_handle* h) {
    const qs_config& c = h->cfg;
    StepParams<Real> p;
    p.pool = h->pool;
    p.n = c.n_envs;
    p.env_id_offset = c.env_id_offset;
    if (h->range_count > 0) {   // a sub-range of whole warp tiles: the tile-major pool makes it a plain pointer offset
        p.pool = static_cast<unsigned char*>(h->pool) + (h->range_first / 32) * (h->bytes_per_env * 32);
        p.n = h->range_count;
        p.env_id_offset = c.env_id_offset + h->range_first;
    }
    p.mom_partial = h->mom_out ? h->mom_scratch : nullptr;
    p.mom_stats = h->mom_stats;
    p.mom_prev = h->mom_out;
    p.ls_tables = h->ls_tables;
    p.ls_counters = h->ls_counters;
    p.ls_steps = h->ls_steps;
    p.substeps = c.substeps;
    p.obs_scaled = c.obs_scaled;
    p.scale_f32 = c.action_scale_f32;
    p.auto_reset = c.auto_reset;
    p.seed = c.seed;
    p.rtol = c.lsoda_rtol;
    p.atol = c.lsoda_atol;
    Model<Real>& m = p.model;
    m.mass = (Real)c.mass;
    m.inv_mass = (Real)(1.0 / c.mass);
    m.g = (Real)c.g;
    m.dt = (Real)c.dt;
    m.I00 = (Real)c.inertia[0]; m.I02 = (Real)c.inertia[2]; m.I11 = (Real)c.inertia[4];
    m.I20 = (Real)c.inertia[6]; m.I22 = (Real)c.inertia[8];
    m.J00 = (Real)c.inv_inertia[0]; m.J02 = (Real)c.inv_inertia[2]; m.J11 = (Real)c.inv_inertia[4];
    m.J20 = (Real)c.inv_inertia[6]; m.J22 = (Real)c.inv_inertia[8];
    for (int i = 0; i < 16; ++i) { m.mix[i] = (Real)c.mix[i]; m.inv_mix[i] = (Real)c.inv_mix[i]; }
    m.tmax = (Real)c.max_prop_thrust;
    m.tmin = (Real)c.min_prop_thrust;
    for (int i = 0; i < QS_TRIG_TAB; ++i) { p.rc.sin_tab[i] = c.sin_tab[i]; p.rc.cos_tab[i] = c.cos_tab[i]; }
    p.dyn = h->dyn_on ? static_cast<Real*>(h->dyn) + (h->range_count > 0 ? h->range_first : 0) : nullptr;   // planes: offset like the pool
    p.dyn_stride = h->dyn_stride;
    p.dr = h->dyn_cfg;
    return p;
}

// Which kernel variant a handle runs: ENV_V1, ENV_V2 (one waypoint, as shipped) or ENV_V2M (v2 with 2-3 waypoints).
inline int env_variant(const qs_handle* h) {
    return h->cfg.env_version == 2 ? (h->cfg.v2_random_waypoints ? ENV_V2M : ENV_V2) : ENV_V1;
}
// Run `body` with `constexpr int VER` bound to the handle's variant.
#define QS_FOR_VARIANT(h, ...)                                                        \
    do {                                                                              \
        switch (qs::env_variant(h)) {                                                 \
            case qs::ENV_V2: { constexpr int VER = qs::ENV_V2; __VA_ARGS__ } break;   \
            case qs::ENV_V2M: { constexpr int VER = qs::ENV_V2M; __VA_ARGS__ } break; \
            default: { constexpr int VER = qs::ENV_V1; __VA_ARGS__ } break;           \
        }                                                                             \
    } while (0)

// Persistent grid: enough CTAs to fill every SM at the kernel's occupancy, never more than the work needs.
template <typename Kernel>
inline unsigned step_grid(const qs_handle* h, Kernel k, int block) {
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, block, 0);
    if (per_sm < 1) per_sm = 1;
    const int64_t need = ((h->range_count > 0 ? h->range_count : h->cfg.n_envs) + block - 1) / block;
    const int64_t cap = (int64_t)per_sm * h->num_sms;
    return (unsigned)(need < cap ? need : cap);
}
}  // namespace qs
