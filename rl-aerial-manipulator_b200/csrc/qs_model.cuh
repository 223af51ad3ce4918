// qs_model.cuh -- rigid-body model of the reference quadrotor: constants, state derivative, mixer, RK4.
//
// Written for sm_100a device code; every function is also __host__ so tests/host_harness can compile
// the very same source with g++ and check it on the CPU-only build box.
//
// Reference semantics (paths relative to the reference root):
//   simul_files/model/params.py:10-36        constants
//   simul_files/model/quadcopter.py:66-103   state_dot
//   simul_files/model/quadcopter.py:105-112  mixer + per-prop clamp
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define QS_HD __host__ __device__ __forceinline__
#else
#define QS_HD inline
#endif

namespace qs {

// Model constants in the arithmetic type of the kernel.  Filled on the host from qs_config (doubles that
// NumPy computed), so the f64 kernels use bit-identical invA / invI to the reference.
template <typename Real>
struct Model {
    Real mass, inv_mass, g, dt;
    Real I00, I02, I11, I20, I22;   // inertia (the reference's I has zeros at 01,10,12,21)
    Real J00, J02, J11, J20, J22;   // inverse inertia (same sparsity)
    Real mix[16], inv_mix[16];
    Real tmax, tmin;                // per-prop thrust clamp
};

template <typename Real> QS_HD Real qs_sqrt(Real x);
template <> QS_HD float qs_sqrt<float>(float x) { return sqrtf(x); }
template <> QS_HD double qs_sqrt<double>(double x) { return sqrt(x); }

// 1/x: exact division in float64 and on the host; in float32 device code MUFU.RCP + one Newton step (__frcp_rn), which
// keeps the IEEE-division slow path (FCHK + call) out of the four-stage RK4 loop
template <typename Real> QS_HD Real qs_rcp(Real x) { return Real(1) / x; }
#if defined(__CUDA_ARCH__) && !defined(QS_EXACT_F32_DIV)
template <> QS_HD float qs_rcp<float>(float x) { return __frcp_rn(x); }
#endif

template <typename Real> QS_HD Real qs_min(Real a, Real b) { return a < b ? a : b; }
template <typename Real> QS_HD Real qs_max(Real a, Real b) { return a > b ? a : b; }

// d/dt [pos, vel, quat(wxyz), omega].  F is the clamped total thrust, M the clamped body moments.
// Thrust acts along the third row of the rotation matrix of the NORMALISED quaternion
// (wRb . [0,0,F] in quadcopter.py:70-74); the quaternion kinematics use the raw quaternion plus the
// norm-restoring term 2*(1-|q|^2)*q (quadcopter.py:77-82).
//
// AXIS_ANGLE selects how that row is evaluated:
//   false  closed form 2(xz-wy), 2(yz+wx), 1-2(x^2+y^2) of q/|q|  -- one division, no transcendental
//   true   the reference's own route (quaternion.py:46-77): theta = 2*arccos(qw/|q|), v = q_xyz/|q_xyz|,
//          Rodrigues with cos/sin(theta).  arccos is ill-conditioned near qw = 1, so this form carries
//          ~1e-13 relative noise; LSODA's step control keys on it near hover, which is why the parity
//          integrator must reproduce the route and not just the value.
//
// WIND (dynamics randomisation): aw is a constant acceleration added to dy[3..5] (the episode's wind force over the true mass).
template <typename Real, bool AXIS_ANGLE = false, bool WIND = false>
QS_HD void state_dot(const Model<Real>& m, const Real* y, Real F, const Real* M, Real* dy, const Real* aw = nullptr) {
    const Real qw = y[6], qx = y[7], qy = y[8], qz = y[9];
    const Real p = y[10], q = y[11], r = y[12];
    const Real n2 = ((qw * qw + qx * qx) + qy * qy) + qz * qz;
    dy[0] = y[3];
    dy[1] = y[4];
    dy[2] = y[5];
    if (AXIS_ANGLE) {
        const double nrm = sqrt((double)n2);
        const double theta = 2.0 * acos((double)qw / nrm);
        const double len = sqrt((double)((qx * qx + qy * qy) + qz * qz));
        double v0 = (double)qx, v1 = (double)qy, v2 = (double)qz;
        if (len > 0.0) { v0 /= len; v1 /= len; v2 /= len; }
        const double c = cos(theta), s = sin(theta);
        const double r20 = v2 * v0 * (1. - c) - v1 * s;
        const double r21 = v2 * v1 * (1. - c) + v0 * s;
        const double r22 = v2 * v2 * (1. - c) + c;
        const double im = 1.0 / (double)m.mass;
        dy[3] = (Real)(im * (r20 * (double)F));
        dy[4] = (Real)(im * (r21 * (double)F));
        dy[5] = (Real)(im * (r22 * (double)F - (double)m.mass * (double)m.g));
    } else {
        const Real inv_n2 = qs_rcp<Real>(n2);
        const Real fm = F * m.inv_mass;
        dy[3] = (Real(2) * (qx * qz - qw * qy) * inv_n2) * fm;
        dy[4] = (Real(2) * (qy * qz + qw * qx) * inv_n2) * fm;
        dy[5] = (Real(1) - Real(2) * (qx * qx + qy * qy) * inv_n2) * fm - m.g;
        if constexpr (WIND) { dy[3] += aw[0]; dy[4] += aw[1]; dy[5] += aw[2]; }
    }
    const Real qerr = Real(2) * (Real(1) - n2);
    dy[6] = Real(-0.5) * (-p * qx - q * qy - r * qz) + qerr * qw;
    dy[7] = Real(-0.5) * (p * qw - r * qy + q * qz) + qerr * qx;
    dy[8] = Real(-0.5) * (q * qw + r * qx - p * qz) + qerr * qy;
    dy[9] = Real(-0.5) * (r * qw - q * qx + p * qy) + qerr * qz;
    // I and inv(I) of the reference have zeros at (0,1),(1,0),(1,2),(2,1); qs_create() rejects anything else
    const Real Iw0 = m.I00 * p + m.I02 * r;
    const Real Iw1 = m.I11 * q;
    const Real Iw2 = m.I20 * p + m.I22 * r;
    const Real t0 = M[0] - (q * Iw2 - r * Iw1);
    const Real t1 = M[1] - (r * Iw0 - p * Iw2);
    const Real t2 = M[2] - (p * Iw1 - q * Iw0);
    dy[10] = m.J00 * t0 + m.J02 * t2;
    dy[11] = m.J11 * t1;
    dy[12] = m.J20 * t0 + m.J22 * t2;
}

// Commanded (F, M) -> per-prop thrusts through invA, clamp, re-mix (quadcopter.py:109-112).
// ETA (dynamics randomisation): prop i delivers eta[i] times its clamped thrust.
template <typename Real, bool ETA = false>
QS_HD void mix_and_clamp(const Model<Real>& m, Real Fcmd, const Real* Mcmd, Real& F, Real* M, const Real* eta = nullptr) {
    Real t[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        Real v = m.inv_mix[4 * i + 0] * Fcmd + m.inv_mix[4 * i + 1] * Mcmd[0] + m.inv_mix[4 * i + 2] * Mcmd[1] +
                 m.inv_mix[4 * i + 3] * Mcmd[2];
        t[i] = qs_max(qs_min(v, m.tmax), m.tmin);
        if constexpr (ETA) t[i] = eta[i] * t[i];
    }
    F = ((t[0] + t[1]) + t[2]) + t[3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
        M[i] = m.mix[4 * (i + 1) + 0] * t[0] + m.mix[4 * (i + 1) + 1] * t[1] + m.mix[4 * (i + 1) + 2] * t[2] +
               m.mix[4 * (i + 1) + 3] * t[3];
}

// Action -> commanded thrust and moments (v2 rl_env_scaledObs.py:125-126, v1 :87-88).
// NumPy >= 2 keeps float32 * python-float products in float32, so with float32 actions the reference
// computes fl32(fl32(a0*fl32(0.18))*fl32(9.81)) and fl32(a_i*fl32(0.1)) and only then widens.
// __fmul_rn forbids FMA contraction so the two roundings really happen.
template <typename Real>
QS_HD void scale_action(const Model<Real>& m, const float* a, int scale_f32, Real& Fcmd, Real* Mcmd) {
    if (scale_f32) {
#if defined(__CUDA_ARCH__)
        const float f = __fmul_rn(__fmul_rn(a[0], (float)m.mass), (float)m.g);
        Fcmd = (Real)f;
        Mcmd[0] = (Real)__fmul_rn(a[1], 0.1f);
        Mcmd[1] = (Real)__fmul_rn(a[2], 0.1f);
        Mcmd[2] = (Real)__fmul_rn(a[3], 0.1f);
#else
        volatile float f1 = a[0] * (float)m.mass;
        volatile float f2 = f1 * (float)m.g;
        Fcmd = (Real)f2;
        for (int i = 0; i < 3; ++i) {
            volatile float mi = a[i + 1] * 0.1f;
            Mcmd[i] = (Real)mi;
        }
#endif
    } else {
        Fcmd = (Real)a[0] * m.mass * m.g;
        Mcmd[0] = (Real)a[1] * Real(0.1);
        Mcmd[1] = (Real)a[2] * Real(0.1);
        Mcmd[2] = (Real)a[3] * Real(0.1);
    }
}

// Classical RK4 over one env step split into `substeps` equal sub-intervals (the throughput integrator;
// the reference uses adaptive LSODA -- see qs_lsoda.cuh for the parity integrator).
// Storage: y, the stage argument, one derivative and the running sum = 4 x 13 Reals live.
// WIND: aw[3] is added to the acceleration of every stage (see state_dot).
template <typename Real, bool WIND = false>
QS_HD void rk4_step(const Model<Real>& m, Real* y, Real F, const Real* M, int substeps, const Real* aw = nullptr) {
    const Real h = m.dt / (Real)substeps;
    const Real h2 = Real(0.5) * h, h6 = h / Real(6), h3 = h / Real(3);
    for (int s = 0; s < substeps; ++s) {
        Real k[13], yt[13], acc[13];
        state_dot<Real, false, WIND>(m, y, F, M, k, aw);
#pragma unroll
        for (int i = 0; i < 13; ++i) { acc[i] = y[i] + h6 * k[i]; yt[i] = y[i] + h2 * k[i]; }
        state_dot<Real, false, WIND>(m, yt, F, M, k, aw);
#pragma unroll
        for (int i = 0; i < 13; ++i) { acc[i] += h3 * k[i]; yt[i] = y[i] + h2 * k[i]; }
        state_dot<Real, false, WIND>(m, yt, F, M, k, aw);
#pragma unroll
        for (int i = 0; i < 13; ++i) { acc[i] += h3 * k[i]; yt[i] = y[i] + h * k[i]; }
        state_dot<Real, false, WIND>(m, yt, F, M, k, aw);
#pragma unroll
        for (int i = 0; i < 13; ++i) y[i] = acc[i] + h6 * k[i];
    }
}

// Dynamics randomisation, per env: d = (k_m, k_I, eta[4], f_wind[3]).  Prop i delivers eta_i times its clamped thrust; the true
// mass m*k_m and inertia k_I*I (inverse J/k_I) are folded into the forces, F' = F/k_m and M' = M/k_I, so that state_dot's thrust
// and rotational terms are the nominal ones: J/k_I*(M - w x k_I*I*w) = J*(M/k_I - w x I*w).  Only the wind acceleration
// aw = f_wind/(m*k_m) stays live through the RK4 stages.
template <typename Real>
QS_HD void dyn_forces(const Model<Real>& m, Real Fcmd, const Real* Mcmd, const Real* d, Real& F, Real* M, Real* aw) {
    mix_and_clamp<Real, true>(m, Fcmd, Mcmd, F, M, d + 2);
    const Real ikm = qs_rcp<Real>(d[0]), ikI = qs_rcp<Real>(d[1]);
    F *= ikm;
    M[0] *= ikI; M[1] *= ikI; M[2] *= ikI;
    const Real im = m.inv_mass * ikm;
    aw[0] = d[6] * im; aw[1] = d[7] * im; aw[2] = d[8] * im;
}

// The same arithmetic with the four stages as a rolled loop (same operations in the same order: acc = y, acc += w_j k_j,
// y_stage = y + c_j k_j): a quarter of the code, for kernels where instruction-cache footprint matters more than loop overhead
// (the fused rollout kernel, csrc/qs_rollout.cu).
template <typename Real>
QS_HD void rk4_step_rolled(const Model<Real>& m, Real* y, Real F, const Real* M, int substeps) {
    const Real h = m.dt / (Real)substeps;
    const Real h2 = Real(0.5) * h, h6 = h / Real(6), h3 = h / Real(3);
    for (int s = 0; s < substeps; ++s) {
        Real k[13], yt[13], acc[13];
#pragma unroll
        for (int i = 0; i < 13; ++i) { acc[i] = y[i]; yt[i] = y[i]; }
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int j = 0; j < 4; ++j) {
            state_dot(m, yt, F, M, k);
            const Real w = (j == 0 || j == 3) ? h6 : h3;
            const Real c = j == 2 ? h : h2;
#pragma unroll
            for (int i = 0; i < 13; ++i) { acc[i] += w * k[i]; yt[i] = y[i] + c * k[i]; }
        }
#pragma unroll
        for (int i = 0; i < 13; ++i) y[i] = acc[i];
    }
}

// state[6:10] /= np.linalg.norm(state[6:10])  (quadcopter.py:114)
template <typename Real>
QS_HD void renormalise_quat(Real* y) {
    const Real n = qs_sqrt<Real>(y[6] * y[6] + y[7] * y[7] + y[8] * y[8] + y[9] * y[9]);
    if (sizeof(Real) == 4) {
        const Real r = qs_rcp<Real>(n);
        y[6] *= r; y[7] *= r; y[8] *= r; y[9] *= r;
    } else {
        y[6] /= n; y[7] /= n; y[8] /= n; y[9] /= n;
    }
}

// ----------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based RNG (Salmon et al. 2011).  counter = (env id lo, env id hi, episode,
// block j), key = seed.  One call yields two 53-bit uniforms in [0,1) built the way NumPy's
// random_sample builds them from two 32-bit words: ((a >> 5) * 2^26 + (b >> 6)) / 2^53.
// ----------------------------------------------------------------------------------------------
QS_HD void mulhilo32(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
    lo = a * b;
    hi = __umulhi(a, b);
#else
    const uint64_t p = (uint64_t)a * (uint64_t)b;
    lo = (uint32_t)p;
    hi = (uint32_t)(p >> 32);
#endif
}

QS_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        mulhilo32(0xD2511F53u, c0, hi0, lo0);
        mulhilo32(0xCD9E8D57u, c2, hi1, lo1);
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

QS_HD double u53(uint32_t a, uint32_t b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// The unit uniforms a reset of (global env id, episode) may consume: v2 with a drawn waypoint count needs 17, everything else
// <= 16.  Kernels generate only the blocks their variant can consume (N = 16 or 18); the test hook returns all QS_N_UNIFORMS.
#define QS_N_UNIFORMS 18
template <int N = QS_N_UNIFORMS>
QS_HD void reset_uniforms(uint64_t seed, uint64_t env_id, uint32_t episode, double* u /*[N]*/) {
    static_assert(N % 2 == 0 && N <= QS_N_UNIFORMS, "two uniforms per Philox block");
#pragma unroll
    for (uint32_t j = 0; j < N / 2; ++j) {
        uint32_t w[4];
        philox4x32_10((uint32_t)env_id, (uint32_t)(env_id >> 32), episode, j, (uint32_t)seed, (uint32_t)(seed >> 32), w);
        u[2 * j] = u53(w[0], w[1]);
        u[2 * j + 1] = u53(w[2], w[3]);
    }
}

}  // namespace qs
