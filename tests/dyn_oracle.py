"""TEST INFRASTRUCTURE ONLY -- CPU oracle of dynamics randomisation (qs_dynamics_randomization), on top of the pinned nominal
oracle (oracle/quad_oracle.py, imported unchanged).

The physics is written in the DIRECT form -- true mass MASS*k_m, inertia k_I*I, inverse INV_INERTIA/k_I, prop i delivering
eta_i times its clamped thrust, a constant world-frame wind force -- not in the kernels' folded form (F/k_m, M/k_I, wind
acceleration), so the parity tests check the algebra of the folding as well as the code.  The action is scaled with the NOMINAL
mass (quad_oracle.scale_action): the controller commands thrust in units of the nominal m*g.
"""
from __future__ import annotations

import numpy as np

from oracle import quad_oracle as qo

N_DYN = 9  # k_m, k_I, eta[4], f_wind[3]


# ---------------------------------------------------------------------------
# the per-episode parameter draw, restated
# ---------------------------------------------------------------------------
def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al. 2011), vectorised: ctr uint32 [...,4], key uint32 [...,2] -> uint32 [...,4]."""
    c = [np.asarray(ctr[..., i], dtype=np.uint64) for i in range(4)]
    k0 = np.asarray(key[..., 0], dtype=np.uint64)
    k1 = np.asarray(key[..., 1], dtype=np.uint64)
    M32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return np.stack(c, axis=-1).astype(np.uint32)


def dynamics_draw(seed, mass_rel, inertia_rel, thrust_rel, wind, env_ids, episodes):
    """[len, N_DYN] parameters (k_m, k_I, eta[4], f_wind[3]) of (global env id, episode): u[0..9] = u53 pairs of Philox4x32-10,
    key = seed, counter = (id lo, id hi, episode, 0x100 + b); k = 1 + rel*(2u - 1), f_wind = wind*(2u - 1), float64."""
    ids = np.asarray(env_ids, dtype=np.uint64).reshape(-1)
    ep = np.asarray(episodes, dtype=np.uint64).reshape(-1)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint32), (len(ids), 2))
    u = np.empty((len(ids), 10))
    for b in range(5):
        ctr = np.stack([ids & np.uint64(0xFFFFFFFF), ids >> np.uint64(32), ep, np.full_like(ids, 0x100 + b)], axis=-1).astype(np.uint32)
        w = philox4x32_10(ctr, key).astype(np.float64)
        u[:, 2 * b] = (np.floor(w[:, 0] / 32) * 67108864.0 + np.floor(w[:, 1] / 64)) * (1.0 / 9007199254740992.0)
        u[:, 2 * b + 1] = (np.floor(w[:, 2] / 32) * 67108864.0 + np.floor(w[:, 3] / 64)) * (1.0 / 9007199254740992.0)
    s = 2.0 * u - 1.0
    d = np.empty((len(ids), N_DYN))
    d[:, 0] = 1.0 + mass_rel * s[:, 0]
    d[:, 1] = 1.0 + inertia_rel * s[:, 1]
    d[:, 2:6] = 1.0 + thrust_rel * s[:, 2:6]
    d[:, 6:9] = wind * s[:, 6:9]
    return d


def dyn_kwargs(d):
    """[N, N_DYN] parameter rows -> the mass_scale / inertia_scale / thrust_scale / wind keywords of physics_update / step."""
    d = np.asarray(d, dtype=np.float64)
    return dict(mass_scale=d[:, 0], inertia_scale=d[:, 1], thrust_scale=d[:, 2:6], wind=d[:, 6:9])


# ---------------------------------------------------------------------------
# physics of the randomised airframe (None = nominal value of that parameter)
# ---------------------------------------------------------------------------
def state_dot(y, F, M, mass_scale=None, inertia_scale=None, wind=None):
    """d/dt of [pos, vel, quat(wxyz), omega] for true mass MASS*k_m, inertia k_I*I and a wind force f_w (world frame, N)."""
    y = np.asarray(y, dtype=np.float64)
    shp = y.shape[:-1]
    k_m = np.broadcast_to(np.ones(shp) if mass_scale is None else np.asarray(mass_scale, dtype=np.float64), shp)
    k_I = np.broadcast_to(np.ones(shp) if inertia_scale is None else np.asarray(inertia_scale, dtype=np.float64), shp)
    f_w = np.broadcast_to(np.zeros(shp + (3,)) if wind is None else np.asarray(wind, dtype=np.float64), shp + (3,))
    mass = qo.MASS * k_m
    qw, qx, qy, qz = y[..., 6], y[..., 7], y[..., 8], y[..., 9]
    p, q, r = y[..., 10], y[..., 11], y[..., 12]
    n2 = qw * qw + qx * qx + qy * qy + qz * qz
    inv_n = 1.0 / np.sqrt(n2)
    w, x, yy, z = qw * inv_n, qx * inv_n, qy * inv_n, qz * inv_n
    out = np.empty_like(y)
    out[..., 0:3] = y[..., 3:6]
    out[..., 3] = (2.0 * (x * z - w * yy)) * F / mass + f_w[..., 0] / mass
    out[..., 4] = (2.0 * (yy * z + w * x)) * F / mass + f_w[..., 1] / mass
    out[..., 5] = (1.0 - 2.0 * (x * x + yy * yy)) * F / mass - qo.GRAV + f_w[..., 2] / mass
    qerr = 2.0 * (1.0 - n2)
    out[..., 6] = -0.5 * (-p * qx - q * qy - r * qz) + qerr * qw
    out[..., 7] = -0.5 * (p * qw - r * qy + q * qz) + qerr * qx
    out[..., 8] = -0.5 * (q * qw + r * qx - p * qz) + qerr * qy
    out[..., 9] = -0.5 * (r * qw - q * qx + p * qy) + qerr * qz
    I = qo.INERTIA
    Iw0 = k_I * (I[0, 0] * p + I[0, 1] * q + I[0, 2] * r)
    Iw1 = k_I * (I[1, 0] * p + I[1, 1] * q + I[1, 2] * r)
    Iw2 = k_I * (I[2, 0] * p + I[2, 1] * q + I[2, 2] * r)
    t0 = M[..., 0] - (q * Iw2 - r * Iw1)
    t1 = M[..., 1] - (r * Iw0 - p * Iw2)
    t2 = M[..., 2] - (p * Iw1 - q * Iw0)
    J = qo.INV_INERTIA
    out[..., 10] = (J[0, 0] * t0 + J[0, 1] * t1 + J[0, 2] * t2) / k_I
    out[..., 11] = (J[1, 0] * t0 + J[1, 1] * t1 + J[1, 2] * t2) / k_I
    out[..., 12] = (J[2, 0] * t0 + J[2, 1] * t1 + J[2, 2] * t2) / k_I
    return out


def mix_and_clamp(F, M, thrust_scale=None):
    """quad_oracle.mix_and_clamp, then prop i delivers thrust_scale[..., i] times its clamped thrust; F and M re-mixed."""
    _, _, t = qo.mix_and_clamp(F, M)
    if thrust_scale is not None:
        t = np.asarray(thrust_scale, dtype=np.float64) * t
    Fc = ((t[..., 0] + t[..., 1]) + t[..., 2]) + t[..., 3]
    Mc = t @ qo.MIX[1:].T
    return Fc, Mc, t


def integrate_rk4(y, F, M, dt=qo.DT, substeps=1, **dyn):
    """Classical RK4 with `substeps` sub-intervals (quad_oracle.integrate_rk4) on the randomised state_dot."""
    y = np.array(y, dtype=np.float64)
    h = dt / substeps
    for _ in range(substeps):
        k1 = state_dot(y, F, M, **dyn)
        k2 = state_dot(y + (0.5 * h) * k1, F, M, **dyn)
        k3 = state_dot(y + (0.5 * h) * k2, F, M, **dyn)
        k4 = state_dot(y + h * k3, F, M, **dyn)
        y = y + (h / 6.0) * (k1 + 2.0 * k2 + 2.0 * k3 + k4)
    return y


def physics_update(y, actions, substeps=1, action_f32=True, mass_scale=None, inertia_scale=None, thrust_scale=None, wind=None):
    """Quadcopter.update of the randomised airframe (RK4): nominal action scaling, mixer with eta, integrate, renormalise."""
    F, M = qo.scale_action(actions, action_f32)
    Fc, Mc, _ = mix_and_clamp(F, M, thrust_scale)
    y2 = integrate_rk4(y, Fc, Mc, substeps=substeps, mass_scale=mass_scale, inertia_scale=inertia_scale, wind=wind)
    qn = np.sqrt(np.sum(y2[..., 6:10] ** 2, axis=-1, keepdims=True))
    y2[..., 6:10] = y2[..., 6:10] / qn
    return y2


def step(b: qo.EnvBatch, actions, substeps=1, action_f32=True, **dyn):
    """quad_oracle.step (no auto-reset) on the randomised airframe; dyn: the keywords of physics_update."""
    b.y = physics_update(b.y, actions, substeps, action_f32, **dyn)
    return qo.step_logic(b)
