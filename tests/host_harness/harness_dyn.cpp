// TEST INFRASTRUCTURE ONLY -- the dynamics-randomisation path of the product's __host__ __device__ headers (csrc/*.cuh),
// compiled with g++: the per-episode draw and one randomised RK4 env step mirroring env_step_kernel<..., DYN = true>'s
// per-thread body.  Builds on harness.cpp (model constants, state load / unload, hh_configure) in a library of its own.
#include "harness.cpp"

template <typename Real, int VER>
static void host_step_dyn(const Model<Real>& m, int substeps, int scale_f32, int obs_scaled, double* y, double* wp, int* ints, double* reals,
                          const float* act, float* obs, double* reward, int* flags, int* ep_len, const double* dyn) {
    EnvState<Real, VER> s;
    load<Real, VER>(s, y, wp, ints[0], ints[1], ints[5] ? reals[0] : (0.0 / 0.0), ints[2], ints[3], ints[4], reals[1], reals[2], ints[6]);
    Real Fcmd, Mcmd[3], F, M[3], d[N_DYN], aw[3];
    for (int k = 0; k < N_DYN; ++k) d[k] = (Real)dyn[k];
    scale_action<Real>(m, act, scale_f32, Fcmd, Mcmd);
    dyn_forces<Real>(m, Fcmd, Mcmd, d, F, M, aw);
    rk4_step<Real, true>(m, s.y, F, M, substeps, aw);
    renormalise_quat<Real>(s.y);
    Real rew;
    const uint32_t fl = step_logic<Real, VER>(s, rew, *ep_len);
    s.ep_ret += rew;
    make_obs<Real, VER>(s, obs_scaled, obs);
    *reward = (double)rew;
    *flags = (int)fl;
    unload<Real, VER>(s, y, wp, ints, reals);
}

extern "C" {

// version 3 = v2 with 2-3 waypoints (ENV_V2M); dyn = (k_m, k_I, eta[4], f_wind[3])
void hh_step_dyn(int version, int f32, int substeps, int scale_f32, int obs_scaled, double* y, double* wp, int* ints, double* reals,
                 const float* act, float* obs, double* reward, int* flags, int* ep_len, const double* dyn) {
    if (version == 3) {
        if (f32) host_step_dyn<float, ENV_V2M>(g_model_f, substeps, scale_f32, obs_scaled, y, wp, ints, reals, act, obs, reward, flags, ep_len, dyn);
        else host_step_dyn<double, ENV_V2M>(g_model_d, substeps, scale_f32, obs_scaled, y, wp, ints, reals, act, obs, reward, flags, ep_len, dyn);
    } else if (version == 2) {
        if (f32) host_step_dyn<float, ENV_V2>(g_model_f, substeps, scale_f32, obs_scaled, y, wp, ints, reals, act, obs, reward, flags, ep_len, dyn);
        else host_step_dyn<double, ENV_V2>(g_model_d, substeps, scale_f32, obs_scaled, y, wp, ints, reals, act, obs, reward, flags, ep_len, dyn);
    } else {
        if (f32) host_step_dyn<float, ENV_V1>(g_model_f, substeps, scale_f32, obs_scaled, y, wp, ints, reals, act, obs, reward, flags, ep_len, dyn);
        else host_step_dyn<double, ENV_V1>(g_model_d, substeps, scale_f32, obs_scaled, y, wp, ints, reals, act, obs, reward, flags, ep_len, dyn);
    }
}

// the dynamics-randomisation draw of (global env id, episode): ranges = mass_rel, inertia_rel, thrust_rel, wind
void hh_dyn_draw(uint64_t seed, const double* ranges, uint64_t env_gid, uint32_t episode, double* out /*[N_DYN]*/) {
    DynRand r;
    r.seed = seed; r.mass_rel = ranges[0]; r.inertia_rel = ranges[1]; r.thrust_rel = ranges[2]; r.wind = ranges[3];
    dyn_draw(r, env_gid, episode, out);
}

}  // extern "C"
