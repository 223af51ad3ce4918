"""ctypes binding of libquadsim.so (include/quadsim.h).  Torch tensors are the only buffers: every
pointer handed to the library is `tensor.data_ptr()` of a CUDA tensor, every stream a raw cudaStream_t.

There is no CPU fallback: if the shared library is missing (not built) or no B200 is visible, loading /
`qs_create` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .quad_constants import QUAD

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("QS_LIB_PATH") or os.path.join(HERE, "lib", "libquadsim.so")

QS_ABI_VERSION = 3
QS_F32, QS_F64 = 0, 1
QS_RK4, QS_LSODA = 0, 1
FLAG_TERMINATED, FLAG_TRUNCATED, FLAG_SUCCESS, FLAG_STOPPED = 0x01, 0x02, 0x04, 0x08
FLAG_CRASHED, FLAG_OOB, FLAG_LSODA_FAIL = 0x10, 0x20, 0x80
MAX_WAYPOINTS = 3
RESET_UNIFORMS = 18
TRIG_TAB = 6


class QsConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("env_version", C.c_int32), ("obs_scaled", C.c_int32), ("precision", C.c_int32),
        ("integrator", C.c_int32), ("substeps", C.c_int32), ("action_scale_f32", C.c_int32), ("auto_reset", C.c_int32),
        ("device", C.c_int32), ("v2_random_waypoints", C.c_int32),
        ("n_envs", C.c_int64), ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
        ("mass", C.c_double), ("g", C.c_double), ("dt", C.c_double),
        ("inertia", C.c_double * 9), ("inv_inertia", C.c_double * 9),
        ("mix", C.c_double * 16), ("inv_mix", C.c_double * 16),
        ("max_prop_thrust", C.c_double), ("min_prop_thrust", C.c_double),
        ("sin_tab", C.c_double * TRIG_TAB), ("cos_tab", C.c_double * TRIG_TAB),
        ("lsoda_rtol", C.c_double), ("lsoda_atol", C.c_double),
    ]


class QsStateView(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in (
        "y", "wp_list", "n_wp", "wp_index", "last_distance", "current_step", "counter", "final_reached",
        "final_yaw", "ep_return", "episode")]


def make_config(env_version=2, n_envs=1, precision="f32", integrator="rk4", substeps=1, obs_scaled=True,
                action_scale_f32=True, auto_reset=True, device=0, env_id_offset=0, seed=0, v2_random_waypoints=False) -> QsConfig:
    """qs_config with the reference's model constants (quad_constants.QUAD) and NumPy-evaluated trig tables."""
    c = QsConfig()
    c.abi_version = QS_ABI_VERSION
    c.env_version = int(env_version)
    c.obs_scaled = int(bool(obs_scaled))
    c.precision = {"f32": QS_F32, "f64": QS_F64}[precision]
    c.integrator = {"rk4": QS_RK4, "lsoda": QS_LSODA}[integrator]
    c.substeps = int(substeps)
    c.action_scale_f32 = int(bool(action_scale_f32))
    c.auto_reset = int(bool(auto_reset))
    c.v2_random_waypoints = int(bool(v2_random_waypoints))
    c.device = int(device)
    c.n_envs = int(n_envs)
    c.env_id_offset = int(env_id_offset)
    c.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    c.mass, c.g, c.dt = QUAD.mass, QUAD.gravity, QUAD.control_dt
    c.inertia[:] = QUAD.inertia.reshape(-1).tolist()
    c.inv_inertia[:] = QUAD.inv_inertia.reshape(-1).tolist()
    c.mix[:] = QUAD.mixer.reshape(-1).tolist()
    c.inv_mix[:] = QUAD.inv_mixer.reshape(-1).tolist()
    c.max_prop_thrust = QUAD.max_total_thrust / 4
    c.min_prop_thrust = QUAD.min_total_thrust / 4
    # v2 trajectory generators (utils2/utils.py:41,84-85): sin(2*t*pi), t = j/K, and cos/sin((j/K) * 2*pi*turns), turns = 1, evaluated
    # with the reference's own NumPy expressions for K = 1 (as shipped, rl_env_scaledObs.py:47) and K = 2, 3 (the :46 alternative)
    for k in (1, 2, 3):
        for j in range(1, k + 1):
            t = j / k
            c.sin_tab[k * (k - 1) // 2 + j - 1] = float(np.sin(2 * t * np.pi))
            c.cos_tab[k * (k - 1) // 2 + j - 1] = float(np.cos((j / k) * (2 * np.pi * 1)))
            assert np.sin(2 * t * np.pi) == np.sin((j / k) * (2 * np.pi * 1))     # one angle per (K, j): the helix shares the sine
    c.lsoda_rtol = c.lsoda_atol = QUAD.odeint_tol
    return c


DYN_PARAMS = 9   # k_m, k_I, eta[4], f_wind[3]


class QsDynamicsRand(C.Structure):
    """qs_dynamics_rand of include/quadsim.h."""
    _fields_ = [("seed", C.c_uint64), ("mass_rel", C.c_double), ("inertia_rel", C.c_double), ("thrust_rel", C.c_double),
                ("wind", C.c_double)]


class QsRolloutArgs(C.Structure):
    """qs_rollout_args of include/quadsim.h."""
    _fields_ = [("policy_image", C.c_void_p), ("obs", C.c_void_p), ("norm_stats", C.c_void_p),
                ("norm_eps", C.c_float), ("norm_clip", C.c_float), ("sample_mode", C.c_int32), ("reserved", C.c_int32),
                ("noise", C.c_void_p), ("noise_seed", C.c_uint64), ("noise_step", C.c_void_p),
                ("clip_lo", C.c_float * 4), ("clip_hi", C.c_float * 4),
                ("obs_norm_out", C.c_void_p), ("actions_out", C.c_void_p), ("actions_clipped_out", C.c_void_p),
                ("values_out", C.c_void_p), ("logp_out", C.c_void_p), ("obs_next", C.c_void_p), ("reward_out", C.c_void_p),
                ("flags_out", C.c_void_p), ("terminal_obs_out", C.c_void_p), ("ep_return_out", C.c_void_p), ("ep_len_out", C.c_void_p)]


SAMPLE_MEAN, SAMPLE_NOISE, SAMPLE_PHILOX = 0, 1, 2


class QsStepManyArgs(C.Structure):
    """qs_step_many_args of include/quadsim.h."""
    _fields_ = [("T", C.c_int32), ("obs_last_only", C.c_int32), ("actions", C.c_void_p), ("action_seed", C.c_uint64),
                ("action_step", C.c_void_p), ("action_lo", C.c_float * 4), ("action_hi", C.c_float * 4),
                ("actions_out", C.c_void_p), ("obs_out", C.c_void_p), ("reward_out", C.c_void_p), ("flags_out", C.c_void_p),
                ("terminal_obs_out", C.c_void_p), ("ep_return_out", C.c_void_p), ("ep_len_out", C.c_void_p)]


class QsPpoHyper(C.Structure):
    """qs_ppo_hyper of include/quadsim.h."""
    _fields_ = [("clip_range", C.c_float), ("ent_coef", C.c_float), ("vf_coef", C.c_float), ("max_grad_norm", C.c_float),
                ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
                ("normalize_advantage", C.c_int32), ("reserved", C.c_int32)]


class QsPidGains(C.Structure):
    """qs_pid_gains of include/quadsim.h (order x, y, z, phi, theta, psi)."""
    _fields_ = [("kp", C.c_double * 6), ("kd", C.c_double * 6), ("ki", C.c_double * 6), ("max_integral", C.c_double)]


_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen libquadsim.so and declare every prototype of include/quadsim.h.  No fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RuntimeError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
    lib = C.CDLL(p)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    lib.qs_abi_version.restype = C.c_int
    lib.qs_last_error.restype = C.c_char_p
    lib.qs_last_error.argtypes = [vp]
    lib.qs_create.argtypes = [C.POINTER(QsConfig), C.POINTER(vp)]
    lib.qs_destroy.argtypes = [vp]
    lib.qs_obs_dim.argtypes = [vp]
    lib.qs_state_bytes_per_env.argtypes = [vp]
    lib.qs_state_bytes_per_env.restype = i64
    lib.qs_reset.argtypes = [vp, vp, vp, vp]
    lib.qs_step.argtypes = [vp] + [vp] * 7 + [vp]
    lib.qs_step_range.argtypes = [vp, i64, i64] + [vp] * 7 + [vp]
    lib.qs_step_range.restype = C.c_int
    lib.qs_step_many.argtypes = [vp, C.POINTER(QsStepManyArgs), vp]
    lib.qs_step_many.restype = C.c_int
    lib.qs_step_moments.argtypes = [vp, vp, vp]
    lib.qs_step_moments_merge.argtypes = [vp, vp]
    lib.qs_step_moments_merge.restype = C.c_int
    lib.qs_step_moments_exchange.argtypes = [vp, vp, vp]
    lib.qs_step_moments_exchange.restype = C.c_int
    lib.qs_get_state.argtypes = [vp, C.POINTER(QsStateView), vp]
    lib.qs_set_state.argtypes = [vp, C.POINTER(QsStateView), vp]
    lib.qs_reset_uniforms.argtypes = [vp, vp, vp, i64, vp, vp]
    lib.qs_lsoda_stats.argtypes = [vp, vp, vp, vp]
    lib.qs_dynamics_randomization.argtypes = [vp, C.POINTER(QsDynamicsRand), vp]
    lib.qs_get_dynamics.argtypes = [vp, vp, vp]
    lib.qs_set_dynamics.argtypes = [vp, vp, vp]
    lib.qs_policy_image_bytes.restype = i64
    lib.qs_policy_prepare.argtypes = [vp, i32, vp, vp]
    lib.qs_policy_prepare.restype = C.c_int
    lib.qs_rollout_step.argtypes = [vp, C.POINTER(QsRolloutArgs), vp]
    lib.qs_rollout_step.restype = C.c_int
    lib.qs_rollout_status.restype = C.c_int
    lib.qs_ppo_default_hyper.argtypes = [C.POINTER(QsPpoHyper)]
    lib.qs_ppo_default_hyper.restype = None
    lib.qs_ppo_n_params.argtypes = [i32]
    lib.qs_ppo_n_params.restype = C.c_int
    lib.qs_ppo_create.argtypes = [i32, i32, C.POINTER(vp)]
    lib.qs_ppo_destroy.argtypes = [vp]
    lib.qs_ppo_update.argtypes = [vp] * 8 + [i64, C.POINTER(QsPpoHyper), vp, vp]
    lib.qs_ppo_grad.argtypes = [vp] * 8 + [i64, C.POINTER(QsPpoHyper), vp, vp, vp]
    lib.qs_ppo_apply.argtypes = [vp, vp, vp, C.POINTER(QsPpoHyper), vp, vp]
    lib.qs_ppo_state.argtypes = [vp] + [C.POINTER(vp)] * 4
    lib.qs_ppo_last_error.restype = C.c_char_p
    for name in ("qs_ppo_create", "qs_ppo_destroy", "qs_ppo_update", "qs_ppo_grad", "qs_ppo_apply", "qs_ppo_state"):
        getattr(lib, name).restype = C.c_int
    lib.qs_pid_default_gains.argtypes = [C.POINTER(QsPidGains)]
    lib.qs_pid_default_gains.restype = None
    lib.qs_pid_run.argtypes = [vp, C.POINTER(QsPidGains), C.c_double] + [vp] * 8 + [i32, vp]
    lib.qs_pid_run.restype = C.c_int
    for name in ("qs_create", "qs_destroy", "qs_obs_dim", "qs_reset", "qs_step", "qs_get_state", "qs_set_state",
                 "qs_reset_uniforms", "qs_lsoda_stats", "qs_step_moments", "qs_dynamics_randomization", "qs_get_dynamics",
                 "qs_set_dynamics"):
        getattr(lib, name).restype = C.c_int
    if lib.qs_abi_version() != QS_ABI_VERSION:
        raise RuntimeError(f"libquadsim ABI {lib.qs_abi_version()} != binding ABI {QS_ABI_VERSION}; rebuild")
    if path is None:
        _lib = lib
    return lib


class QuadsimError(RuntimeError):
    pass


def check(lib, handle, rc: int, what: str) -> None:
    if rc != 0:
        msg = lib.qs_last_error(handle)
        raise QuadsimError(f"{what} failed ({rc}): {msg.decode() if msg else '?'}")
