// qs_env.cuh -- per-env register state of WaypointQuadEnv and everything in step() that is not physics:
// reward, the waypoint / hold / termination state machine, observation, reset.
//
// Reference semantics (paths relative to the reference root):
//   v2  initial-implementation-v2/rl_env_scaledObs.py   step :123-196, reward :198-231, obs :98-121, reset :40-96
//       initial-implementation-v2/utils2/utils.py        trajectories :12-94, euler angles :4-9 (scipy as_euler('xyz'))
//   v1  initial-implementation-v1/rl_env_scaledObs.py   step :85-140, reward :142-168, obs :65-83, reset :32-63
//       initial-implementation-v1/rl_env.py              same with unscaled obs
// Host+device so tests/host_harness can run the same code under g++.
#pragma once
#include "qs_model.cuh"

namespace qs {

// ENV_V2M: v2 with waypoint lists of 2-3 entries (the `randint(2, 4)` alternative of rl_env_scaledObs.py:46); same step logic and
// observation as ENV_V2, a wider state record
enum : int { ENV_V1 = 1, ENV_V2 = 2, ENV_V2M = 3 };
QS_HD constexpr bool is_v2(int ver) { return ver == ENV_V2 || ver == ENV_V2M; }

constexpr uint32_t FLAG_TERMINATED = 0x01, FLAG_TRUNCATED = 0x02, FLAG_SUCCESS = 0x04, FLAG_STOPPED = 0x08,
                   FLAG_CRASHED = 0x10, FLAG_OOB = 0x20, FLAG_LSODA_FAIL = 0x80;

template <int VER> struct EnvTraits;
template <> struct EnvTraits<ENV_V1> { static constexpr int NWP = 2, OBS = 17, MAX_STEPS = 1200; };
template <> struct EnvTraits<ENV_V2> { static constexpr int NWP = 1, OBS = 20, MAX_STEPS = 2000; };
template <> struct EnvTraits<ENV_V2M> { static constexpr int NWP = 3, OBS = 20, MAX_STEPS = 2000; };
constexpr int COUNTER_LIMIT = 500;

// Constants of the episode generator that must be bit-identical to NumPy's (sin/cos of 2*pi*j/K).
struct ResetConsts {
    double sin_tab[6], cos_tab[6];   // index K*(K-1)/2 + j-1 for K = 1..3, j = 1..K
};

// Hidden state of one env, held in registers for the whole step.
//   bits: current_step[0:12) | counter[12:24) | wp_index[24:26) | n_wp[26:28) | final_reached[28] | has_last[29]
template <typename Real, int VER>
struct EnvState {
    static constexpr int NWP = EnvTraits<VER>::NWP;
    Real y[13];
    Real wp[NWP][3];
    Real final_yaw;
    Real last_d;
    Real ep_ret;
    uint32_t bits;
    uint32_t episode;

    QS_HD int step() const { return bits & 0xFFF; }
    QS_HD int counter() const { return (bits >> 12) & 0xFFF; }
    QS_HD int wp_index() const { return (bits >> 24) & 3; }
    QS_HD int n_wp() const { return (bits >> 26) & 3; }
    QS_HD bool final_reached() const { return (bits >> 28) & 1; }
    QS_HD bool has_last() const { return (bits >> 29) & 1; }
    QS_HD void set(int step, int counter, int idx, int nwp, bool fin, bool has_last) {
        step = step > 0xFFF ? 0xFFF : step;
        counter = counter > 0xFFF ? 0xFFF : counter;
        bits = (uint32_t)step | ((uint32_t)counter << 12) | ((uint32_t)idx << 24) | ((uint32_t)nwp << 26) |
               ((uint32_t)fin << 28) | ((uint32_t)has_last << 29);
    }
    // current_waypoint == waypoint_list[min(waypoint_index, len-1)] at all times in the reference:
    // it starts at list[0], moves to list[index] while index < len, and otherwise keeps its last value.
    QS_HD int cur_index() const {
        const int i = wp_index(), n = n_wp();
        return i < n ? i : n - 1;
    }
    QS_HD void cur_wp(Real* out) const {
        const int c = cur_index();
#pragma unroll
        for (int j = 0; j < NWP; ++j)
            if (j == c) { out[0] = wp[j][0]; out[1] = wp[j][1]; out[2] = wp[j][2]; }
    }
};

// ------------------------------------------------------------------------------------------------
// math helpers
// ------------------------------------------------------------------------------------------------
template <typename Real> QS_HD Real qs_atan2(Real y, Real x);
template <> QS_HD float qs_atan2<float>(float y, float x) { return atan2f(y, x); }
template <> QS_HD double qs_atan2<double>(double y, double x) { return atan2(y, x); }
template <typename Real> QS_HD Real qs_hypot(Real y, Real x);
template <> QS_HD float qs_hypot<float>(float y, float x) { return hypotf(y, x); }
template <> QS_HD double qs_hypot<double>(double y, double x) { return hypot(y, x); }
template <typename Real> QS_HD Real qs_abs(Real x) { return x < Real(0) ? -x : x; }

template <typename Real> QS_HD Real norm3(const Real* v) { return qs_sqrt<Real>(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }

// scipy Rotation.from_quat([x,y,z,w]).as_euler('xyz') -- Bernardes & Viollet half-angle form with scipy's
// 1e-7 gimbal-lock window (third angle forced to zero there) and comparison-based wrap to [-pi, pi].
template <typename Real>
QS_HD void quat_to_rpy(const Real* q /*wxyz*/, Real& roll, Real& pitch, Real& yaw) {
    const Real PI = Real(3.141592653589793238462643383279502884);
    const Real n = qs_sqrt<Real>(q[1] * q[1] + q[2] * q[2] + q[3] * q[3] + q[0] * q[0]);
    const Real x = q[1] / n, y = q[2] / n, z = q[3] / n, w = q[0] / n;
    const Real a = w - y, b = x + z, c = y + w, d = z - x;
    const Real half_sum = qs_atan2<Real>(b, a);
    const Real half_diff = qs_atan2<Real>(d, c);
    const Real ang1 = Real(2) * qs_atan2<Real>(qs_hypot<Real>(c, d), qs_hypot<Real>(a, b));
    const bool case1 = qs_abs<Real>(ang1) <= Real(1e-7);
    const bool case2 = qs_abs<Real>(ang1 - PI) <= Real(1e-7);
    if (!(case1 || case2)) {
        roll = half_sum - half_diff;
        yaw = half_sum + half_diff;
    } else {
        roll = case1 ? Real(2) * half_sum : Real(-2) * half_diff;
        yaw = Real(0);
    }
    pitch = ang1 - PI / Real(2);
    const Real TWO_PI = Real(2) * PI;
    roll = roll < -PI ? roll + TWO_PI : (roll > PI ? roll - TWO_PI : roll);
    pitch = pitch < -PI ? pitch + TWO_PI : (pitch > PI ? pitch - TWO_PI : pitch);
    yaw = yaw < -PI ? yaw + TWO_PI : (yaw > PI ? yaw - TWO_PI : yaw);
}

// ------------------------------------------------------------------------------------------------
// observation
// ------------------------------------------------------------------------------------------------
template <typename Real> struct ObsScale;
// float64: true division like the reference (pos / 10.0 ...), then the float32 cast
template <> struct ObsScale<double> {
    static QS_HD float pos(double v) { return (float)(v / 10.0); }
    static QS_HD float vel(double v) { return (float)(v / 5.0); }
    static QS_HD float rel(double v) { return (float)(v / 2.0); }
    static QS_HD float yaw(double v) { return (float)(v / 3.141592653589793); }
};
// float32: reciprocal multiplies (<= 1 ulp from the true quotient)
template <> struct ObsScale<float> {
    static QS_HD float pos(float v) { return v * 0.1f; }
    static QS_HD float vel(float v) { return v * 0.2f; }
    static QS_HD float rel(float v) { return v * 0.5f; }
    static QS_HD float yaw(float v) { return v * 0.31830988618379067f; }
};

template <typename Real, int VER>
QS_HD void make_obs(const EnvState<Real, VER>& s, int obs_scaled, float* obs) {
    using S = ObsScale<Real>;
    constexpr int NWP = EnvState<Real, VER>::NWP;
    Real cw[3];
    s.cur_wp(cw);
    const Real rel[3] = {cw[0] - s.y[0], cw[1] - s.y[1], cw[2] - s.y[2]};
    if (obs_scaled) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            obs[i] = S::pos(s.y[i]);
            obs[3 + i] = S::vel(s.y[3 + i]);
            obs[10 + i] = S::vel(s.y[10 + i]);
            obs[13 + i] = S::rel(rel[i]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            obs[i] = (float)s.y[i];
            obs[3 + i] = (float)s.y[3 + i];
            obs[10 + i] = (float)s.y[10 + i];
            obs[13 + i] = (float)rel[i];
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) obs[6 + i] = (float)s.y[6 + i];
    if (is_v2(VER)) {
        // rel_pos_next = list[index+1] - current_waypoint while index < len-1, else zeros (:104-107)
        Real nx[3] = {Real(0), Real(0), Real(0)};
        const int idx = s.wp_index(), n = s.n_wp();
        if (NWP > 1 && idx < n - 1) {
#pragma unroll
            for (int j = 0; j + 1 < NWP; ++j)
                if (j == idx) { nx[0] = s.wp[j + 1][0] - cw[0]; nx[1] = s.wp[j + 1][1] - cw[1]; nx[2] = s.wp[j + 1][2] - cw[2]; }
        }
        obs[16] = obs_scaled ? S::rel(nx[0]) : (float)nx[0];
        obs[17] = obs_scaled ? S::rel(nx[1]) : (float)nx[1];
        obs[18] = obs_scaled ? S::rel(nx[2]) : (float)nx[2];
        obs[19] = obs_scaled ? S::yaw(s.final_yaw) : (float)s.final_yaw;
    } else {
        // is_final = np.allclose(current_waypoint, waypoint_list[-1])  (value compare, rtol 1e-5, atol 1e-8; :80)
        const int last = s.n_wp() - 1;
        Real lw[3] = {Real(0), Real(0), Real(0)};
#pragma unroll
        for (int j = 0; j < NWP; ++j)
            if (j == last) { lw[0] = s.wp[j][0]; lw[1] = s.wp[j][1]; lw[2] = s.wp[j][2]; }
        bool close = true;
#pragma unroll
        for (int i = 0; i < 3; ++i) close = close && (qs_abs<Real>(cw[i] - lw[i]) <= Real(1e-8) + Real(1e-5) * qs_abs<Real>(lw[i]));
        obs[16] = close ? 1.0f : 0.0f;
    }
}

// ------------------------------------------------------------------------------------------------
// step logic after quadcopter.update(): reward + state machine.  Returns the QS_FLAG_* byte and the
// reward; `ep_len` receives the Monitor-style episode length as of this step.
// ------------------------------------------------------------------------------------------------
template <typename Real, int VER>
QS_HD uint32_t step_logic(EnvState<Real, VER>& s, Real& reward_out, int& ep_len) {
    const Real* pos = s.y;
    const Real* vel = s.y + 3;
    const Real* om = s.y + 10;
    Real cw[3];
    s.cur_wp(cw);
    const Real dv[3] = {pos[0] - cw[0], pos[1] - cw[1], pos[2] - cw[2]};
    const Real d = norm3<Real>(dv);
    const Real vn = norm3<Real>(vel), wn = norm3<Real>(om);

    int step = s.step(), counter = s.counter(), idx = s.wp_index();
    const int nwp = s.n_wp();
    bool fin = s.final_reached();
    const bool fin0 = fin;

    // _calculate_reward (v2 :198-231, v1 :142-168)
    Real dist_r = -d * (is_v2(VER) ? Real(10) : Real(2));
    Real speed = Real(-0.1) * (vn * vn);
    if (wn > Real(0.1)) speed -= Real(0.01) * (wn * wn);
    Real time_pen = Real(-0.1);
    Real prog = Real(0);
    if (s.has_last()) {
        prog = Real(20) * (s.last_d - d);
        if (prog > Real(0)) prog += Real(2);
    }
    s.last_d = d;
    if (is_v2(VER) && fin0) {
        prog = Real(0);
        time_pen = Real(0);
        if (d < Real(0.1)) dist_r = Real(1);
    }
    Real reward = ((dist_r + speed) + time_pen) + prog;

    uint32_t flags = 0;
    bool early = false;
    bool truncated;

    if (is_v2(VER)) {
        truncated = step >= EnvTraits<VER>::MAX_STEPS;   // evaluated before the increment (:144-145)
        step += 1;
        ep_len = step;
        if (d < Real(0.1)) {
            if (!fin0) { idx += 1; reward += Real(100); }
            if (idx < nwp) {
                // next waypoint becomes current; falls through to the crash / bounds checks
            } else {
                Real roll, pitch, yaw;
                quat_to_rpy<Real>(s.y + 6, roll, pitch, yaw);
                const Real TWO_PI = Real(2) * Real(3.141592653589793238462643383279502884);
                const Real dyaw = qs_abs<Real>(yaw - s.final_yaw);
                const bool stopped = (vn < Real(0.1)) && (wn < Real(0.1));
                if (!fin0) {
                    // first arrival at the final waypoint (:156-164)
                    fin = true;
                    const Real stop_b = vn < Real(1) ? Real(150) * (Real(1) - vn * vn) : Real(0);
                    const Real yaw_b = dyaw < TWO_PI ? Real(100) * (Real(1) - dyaw / TWO_PI) : Real(0);
                    reward = ((reward + Real(200)) + stop_b) + yaw_b;
                } else {
                    // hold phase (:165-179)
                    const Real yaw_b = dyaw < TWO_PI ? Real(30) * (Real(1) - dyaw / TWO_PI) : Real(0);
                    const Real ar = qs_abs<Real>(roll), ap = qs_abs<Real>(pitch);
                    const Real roll_b = ar < Real(0.2) ? Real(10) * (Real(1) - ar / Real(0.2)) : Real(-.1) * ar;
                    const Real pit_b = ap < Real(0.2) ? Real(10) * (Real(1) - ap / Real(0.2)) : Real(-.1) * ap;
                    reward = ((reward + yaw_b) + roll_b) + pit_b;
                    if (counter <= COUNTER_LIMIT) counter += 1;
                    else flags |= FLAG_TERMINATED;
                }
                flags |= FLAG_SUCCESS | (stopped ? FLAG_STOPPED : 0u);
                early = true;
            }
        }
        if (!early && fin0) counter += 1;   // `if self.counter_activated: self.counter += 1` (:181-182)
    } else {
        // v1: approach shaping inside 0.5 m (:100-110); NaN direction when exactly on the waypoint -> both tests false
        const Real wd[3] = {cw[0] - pos[0], cw[1] - pos[1], cw[2] - pos[2]};
        const Real wdn = norm3<Real>(wd);
        const Real vt = vel[0] * (wd[0] / wdn) + vel[1] * (wd[1] / wdn) + vel[2] * (wd[2] / wdn);
        if (d < Real(0.5) && vt > Real(0.1)) reward += Real(10);
        else if (d < Real(0.5) && vt < Real(0.1)) reward -= Real(10);
        truncated = false;
        ep_len = step + 1;
        if (d < Real(0.1)) {
            reward += Real(100);
            idx += 1;
            if (idx >= nwp) {
                // all waypoints reached (:117-124): terminated, truncated is the literal False, step not counted
                const Real rot_b = wn < Real(0.1) ? Real(100) : Real(-20) * wn;
                const Real stop_b = vn < Real(0.1) ? Real(100) : Real(-10) * vn;
                reward = ((reward + Real(400)) + stop_b) + rot_b;
                flags |= FLAG_TERMINATED | FLAG_SUCCESS | (vn < Real(0.1) ? FLAG_STOPPED : 0u);
                early = true;
            }
        }
        if (!early) {
            truncated = step >= EnvTraits<VER>::MAX_STEPS;
            step += 1;
        }
    }

    if (!early) {
        if (pos[2] < Real(0.1)) {
            reward -= Real(100);
            if (vel[2] < Real(0)) reward += vel[2] * Real(100);
            flags |= FLAG_TERMINATED | FLAG_CRASHED;
        } else if (norm3<Real>(pos) > Real(10)) {
            reward -= Real(100);
            flags |= FLAG_TERMINATED | FLAG_OOB;
        }
    }
    if (truncated) flags |= FLAG_TRUNCATED;
    if (idx > 3) idx = 3;
    s.set(step, counter, idx, nwp, fin, true);
    reward_out = reward;
    return flags;
}

// ------------------------------------------------------------------------------------------------
// reset: consumes the unit uniforms of (seed, global env id, episode) in the reference's draw order.
//   uniform(lo,hi) = lo + (hi-lo)*u ; rand() = u ; randint(lo,hi) = lo + floor(u*(hi-lo))
// ------------------------------------------------------------------------------------------------
// lo + (hi - lo) * u with the product and the sum rounded separately (NumPy's uniform()); on the device the
// _rn intrinsics keep nvcc from contracting them into one FMA, which would change the last bit.
QS_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
QS_HD double add_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
QS_HD double uniform_rn(double lo, double hi, double u) { return add_rn(lo, mul_rn(hi - lo, u)); }

// ------------------------------------------------------------------------------------------------
// dynamics randomisation: the 9 per-env parameters of an episode, d = (k_m, k_I, eta[4], f_wind[3]) (qs_dynamics_rand).
// u[0..9]: Philox4x32-10 keyed on r.seed, counter = (env id lo, env id hi, episode, 0x100 + b), b = 0..4 -- word 3 never
// meets the reset's blocks (j < 9), so the two streams are independent even under one seed.  Round-to-nearest products and
// sums, in float64: a NumPy restatement reproduces the parameters bit for bit.
// ------------------------------------------------------------------------------------------------
struct DynRand {
    uint64_t seed;
    double mass_rel, inertia_rel, thrust_rel, wind;
};
constexpr int N_DYN = 9;

QS_HD double dyn_sym(double u) { return add_rn(mul_rn(2.0, u), -1.0); }   // 2u - 1 in [-1, 1)

QS_HD void dyn_draw(const DynRand& r, uint64_t env_gid, uint32_t episode, double* d /*[N_DYN]*/) {
    double u[10];
#pragma unroll
    for (uint32_t b = 0; b < 5; ++b) {
        uint32_t w[4];
        philox4x32_10((uint32_t)env_gid, (uint32_t)(env_gid >> 32), episode, 0x100u + b, (uint32_t)r.seed, (uint32_t)(r.seed >> 32), w);
        u[2 * b] = u53(w[0], w[1]);
        u[2 * b + 1] = u53(w[2], w[3]);
    }
    d[0] = add_rn(1.0, mul_rn(r.mass_rel, dyn_sym(u[0])));
    d[1] = add_rn(1.0, mul_rn(r.inertia_rel, dyn_sym(u[1])));
#pragma unroll
    for (int i = 0; i < 4; ++i) d[2 + i] = add_rn(1.0, mul_rn(r.thrust_rel, dyn_sym(u[2 + i])));
#pragma unroll
    for (int j = 0; j < 3; ++j) d[6 + j] = mul_rn(r.wind, dyn_sym(u[6 + j]));
}

template <typename Real, int VER>
QS_HD void reset_env(EnvState<Real, VER>& s, const ResetConsts& rc, uint64_t seed, uint64_t env_gid) {
    constexpr int NWP = EnvState<Real, VER>::NWP;
    const double PI = 3.141592653589793;
    constexpr int NU = VER == ENV_V2M ? 18 : 16;
    double u[NU];
    reset_uniforms<NU>(seed, env_gid, s.episode, u);
    int k = 0;
    double start[3];
    start[0] = uniform_rn(-1.0, 1.0, u[k++]);
    start[1] = uniform_rn(-1.0, 1.0, u[k++]);
    k++;                                  // third component of uniform(-1,1,3): drawn, then overwritten
    start[2] = uniform_rn(1.0, 2.0, u[k++]);
#pragma unroll
    for (int i = 0; i < 13; ++i) s.y[i] = Real(0);
    s.y[0] = (Real)start[0];
    s.y[1] = (Real)start[1];
    s.y[2] = (Real)start[2];
    s.y[6] = Real(1);                     // attitude (0,0,0)  (quadcopter.py:25-38)
    s.last_d = Real(0);
    s.ep_ret = Real(0);
    s.final_yaw = Real(0);
#pragma unroll
    for (int j = 0; j < NWP; ++j) { s.wp[j][0] = Real(0); s.wp[j][1] = Real(0); s.wp[j][2] = Real(0); }
    int nwp = 1;
    if (is_v2(VER)) {
        if (VER == ENV_V2M) nwp = 2 + (int)floor(u[k++] * 2.0);    // num_waypoints = randint(2, 4), drawn where :46 has it
        k += 4;                           // roll, pitch, yaw draws and `rand() < 0`: consumed, unused (:49-52)
        int kind;
        if (u[k++] < 0.3) kind = 0;       // linear
        else if (u[k++] < 0.6) kind = 1;  // curved
        else kind = 2;                    // helical
        const int tb = nwp * (nwp - 1) / 2;                          // this K's row of the sin/cos tables
        double end[3] = {0.0, 0.0, 0.0};
        int axis = -1;
        if (kind <= 1) {
            end[0] = uniform_rn(-1.0, 1.0, u[k++]);
            end[1] = uniform_rn(-1.0, 1.0, u[k++]);
            k++;
            end[2] = uniform_rn(0.5, 3.0, u[k++]);
            if (kind == 1) axis = 2 - (int)floor(u[k++] * 3.0);     // randint(0,3): 0 -> z, 1 -> y, 2 -> x
        }
#pragma unroll
        for (int j = 0; j < NWP; ++j) {
            if (j < nwp) {
                double w[3];
                if (kind <= 1) {
                    const double t = (double)(j + 1) / (double)nwp;  // i / num_waypoints, i = 1..K (utils.py:19,37)
#pragma unroll
                    for (int i = 0; i < 3; ++i) {
                        w[i] = add_rn(start[i], mul_rn(t, end[i] - start[i]));
                        if (kind == 1 && i == axis) w[i] = add_rn(w[i], rc.sin_tab[tb + j]);   // + sin(2*t*pi)
                    }
                    if (kind == 1) w[2] = fmax(w[2], 0.2);
                } else {
                    w[0] = add_rn(start[0], mul_rn(0.8, rc.cos_tab[tb + j]));
                    w[1] = add_rn(start[1], mul_rn(0.8, rc.sin_tab[tb + j]));
                    w[2] = fmax(add_rn(start[2], mul_rn((double)(j + 1), 0.4)), 0.2);
                }
                s.wp[j][0] = (Real)w[0];
                s.wp[j][1] = (Real)w[1];
                s.wp[j][2] = (Real)w[2];
            }
        }
        s.final_yaw = (Real)uniform_rn(-PI, PI, u[k++]);
    } else {
        nwp = 1 + (int)floor(u[k++] * 2.0);                         // randint(1,3)
#pragma unroll
        for (int j = 0; j < NWP; ++j) {
            if (j < nwp) {
                s.wp[j][0] = (Real)uniform_rn(-1.0, 1.0, u[k++]);
                s.wp[j][1] = (Real)uniform_rn(-1.0, 1.0, u[k++]);
                s.wp[j][2] = (Real)uniform_rn(1.0, 3.0, u[k++]);
            }
        }
    }
    s.set(0, 0, 0, nwp, false, false);
}

}  // namespace qs
