"""Test helper: builds tests/host_harness/harness_dyn.cpp with g++ (the dynamics-randomisation path of the product's
__host__ __device__ headers, compiled for the CPU) and wraps it with ctypes.  Test infrastructure only."""
import ctypes as C
import os
import subprocess

import numpy as np

from harness_util import CSRC, ROOT, HostHarness, ptr

SRC = os.path.join(ROOT, "tests", "host_harness", "harness_dyn.cpp")
OUT = os.path.join(ROOT, "build", "libqs_host_dyn.so")


def build_dyn_harness() -> str:
    deps = [SRC, os.path.join(ROOT, "tests", "host_harness", "harness.cpp")] + \
        [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in deps):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        # -ffp-contract=off: products and sums round separately, as in the NumPy oracle
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", SRC, "-o", OUT])
    return OUT


class DynHarness(HostHarness):
    """HostHarness (reset, uniforms, nominal step, ...) plus the randomised step and the parameter draw."""

    def __init__(self, cfg):
        self.lib = C.CDLL(build_dyn_harness())
        self.lib.hh_configure(C.byref(cfg))
        self.cfg = cfg
        L = self.lib
        L.hh_reset.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_int] + [C.c_void_p] * 5
        L.hh_uniforms.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]
        L.hh_step_dyn.argtypes = [C.c_int] * 5 + [C.c_void_p] * 10
        L.hh_dyn_draw.argtypes = [C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]

    def step_dyn(self, version, st, act, dyn, f32=False, substeps=1, scale_f32=True, obs_scaled=True):
        """One randomised RK4 env step (no auto-reset) from state dict `st`; dyn = (k_m, k_I, eta[4], f_wind[3])."""
        y = np.array(st["y"], dtype=np.float64)
        wp = np.zeros(9)
        wp[:] = np.asarray(st["wp_list"], dtype=np.float64).reshape(-1)[:9]
        ld = st["last_distance"]
        has_last = not (ld is None or np.isnan(ld))
        ints = np.array([st["n_wp"], st["wp_index"], st["current_step"], st.get("counter", 0),
                         int(st.get("final_reached", False)), int(has_last), st.get("episode", 0)], dtype=np.int32)
        reals = np.array([ld if has_last else 0.0, st.get("final_yaw", 0.0), st.get("ep_return", 0.0)], dtype=np.float64)
        act = np.ascontiguousarray(act, dtype=np.float32)
        dyn = np.ascontiguousarray(dyn, dtype=np.float64)
        obs = np.zeros(20 if version in (2, 3) else 17, dtype=np.float32)
        rew, flags, ep_len = C.c_double(), C.c_int(), C.c_int()
        self.lib.hh_step_dyn(version, int(f32), substeps, int(scale_f32), int(obs_scaled), ptr(y), ptr(wp), ptr(ints), ptr(reals),
                             ptr(act), ptr(obs), C.byref(rew), C.byref(flags), C.byref(ep_len), ptr(dyn))
        out = dict(y=y, wp_list=wp.reshape(3, 3), n_wp=int(ints[0]), wp_index=int(ints[1]), current_step=int(ints[2]),
                   counter=int(ints[3]), final_reached=bool(ints[4]), last_distance=reals[0] if ints[5] else np.nan,
                   final_yaw=reals[1], ep_return=reals[2])
        return out, obs, rew.value, flags.value, ep_len.value

    def dyn_draw(self, seed, ranges, env_gid, episode):
        """The 9 dynamics-randomisation parameters of (global env id, episode); ranges = mass, inertia, thrust, wind."""
        r = np.ascontiguousarray(ranges, dtype=np.float64)
        out = np.zeros(9)
        self.lib.hh_dyn_draw(seed, ptr(r), env_gid, episode, ptr(out))
        return out
