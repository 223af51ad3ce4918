"""BatchedQuadEnv -- native tensor API over libquadsim (one handle = one shard of envs on one B200).

This is the throughput surface: every input and output is a torch CUDA tensor, nothing is copied to the
host, and calls are ordered on the current torch CUDA stream.  The SB3-compatible NumPy surface
(`reset / step_async / step_wait`, `infos` dicts) is `vec_env.QuadVecEnv`, built on top of this class.

Replaces, for N envs at once (reference root-relative paths):
    WaypointQuadEnv.reset / step   initial-implementation-v2/rl_env_scaledObs.py:40-231
                                   initial-implementation-v1/rl_env_scaledObs.py:32-168, rl_env.py
    Quadcopter.update              simul_files/model/quadcopter.py:105-114
    DummyVecEnv auto-reset         (stable_baselines3, call site initial-implementation-v1/rl_train_vecN.py:10)
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

from . import _cabi
from ._cabi import QsStateView, check, load_library, make_config

OBS_DIM = {1: 17, 2: 20}

_STATE_FIELDS = {
    "y": (torch.float64, (13,)), "wp_list": (torch.float64, (3, 3)), "n_wp": (torch.int32, ()),
    "wp_index": (torch.int32, ()), "last_distance": (torch.float64, ()), "current_step": (torch.int32, ()),
    "counter": (torch.int32, ()), "final_reached": (torch.uint8, ()), "final_yaw": (torch.float64, ()),
    "ep_return": (torch.float64, ()), "episode": (torch.int32, ()),
}


@dataclass
class StepOut:
    obs: torch.Tensor            # f32[n, obs_dim]; reset obs for envs that finished (auto_reset)
    reward: torch.Tensor         # f32[n] or f64[n]
    flags: torch.Tensor          # u8[n], QS_FLAG_* bits
    terminal_obs: torch.Tensor   # f32[n, obs_dim]; rows valid where done
    ep_return: torch.Tensor      # rows valid where done
    ep_len: torch.Tensor         # i32[n]; rows valid where done

    @property
    def done(self) -> torch.Tensor:
        return (self.flags & 3) != 0

    @property
    def terminated(self) -> torch.Tensor:
        return (self.flags & _cabi.FLAG_TERMINATED) != 0

    @property
    def truncated(self) -> torch.Tensor:
        return (self.flags & _cabi.FLAG_TRUNCATED) != 0


class BatchedQuadEnv:
    """N independent WaypointQuadEnv instances stepped by one fused sm_100a kernel.

    v2_random_waypoints (env_version 2): False = `num_waypoints = 1` as the reference ships it (rl_env_scaledObs.py:47); True = the
    `np.random.randint(2, 4)` alternative it keeps commented out at :46 -- trajectories of 2 or 3 waypoints.

    dynamics_randomization (RK4 only): None = the nominal airframe, or a dict {"mass", "inertia", "thrust", "wind"[, "seed"]} --
    every episode of every env then draws its own true mass mass*(1 +- mass), inertia I*(1 +- inertia), per-prop thrust factors
    1 +- thrust and a constant world-frame wind force of up to +-wind N per axis (uniform; seed defaults to the env seed).  The
    action scaling keeps the nominal mass.  See `randomize_dynamics`, `dynamics`, `set_dynamics`."""

    def __init__(self, n_envs: int, env_version: int = 2, precision: str = "f32", integrator: str = "rk4",
                 substeps: int = 1, obs_scaled: bool = True, action_scale_f32: bool = True, auto_reset: bool = True,
                 device: int | torch.device | None = None, env_id_offset: int = 0, seed: int = 0,
                 v2_random_waypoints: bool = False, dynamics_randomization: dict | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedQuadEnv needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device if isinstance(device, int) else (device.index or 0))
        self.lib = load_library()
        self.cfg = make_config(env_version=env_version, n_envs=n_envs, precision=precision, integrator=integrator,
                               substeps=substeps, obs_scaled=obs_scaled, action_scale_f32=action_scale_f32,
                               auto_reset=auto_reset, device=self.device.index, env_id_offset=env_id_offset, seed=seed,
                               v2_random_waypoints=v2_random_waypoints)
        self.n_envs = int(n_envs)
        self.env_version = int(env_version)
        self.obs_dim = OBS_DIM[self.env_version]
        self.precision = precision
        self.integrator = integrator
        self.real_dtype = torch.float32 if precision == "f32" else torch.float64
        self._h = C.c_void_p()
        check(self.lib, None, self.lib.qs_create(C.byref(self.cfg), C.byref(self._h)), "qs_create")
        n, d = self.n_envs, self.obs_dim
        dev = self.device
        # persistent output buffers (caller-owned from the library's point of view)
        self.obs = torch.empty((n, d), dtype=torch.float32, device=dev)
        self.reward = torch.empty((n,), dtype=self.real_dtype, device=dev)
        self.flags = torch.zeros((n,), dtype=torch.uint8, device=dev)
        self.terminal_obs = torch.zeros((n, d), dtype=torch.float32, device=dev)
        self.ep_return = torch.zeros((n,), dtype=self.real_dtype, device=dev)
        self.ep_len = torch.zeros((n,), dtype=torch.int32, device=dev)
        self.seed = int(seed)
        self.dynamics_randomization = None
        if dynamics_randomization is not None:
            self.randomize_dynamics(dynamics_randomization)

    # -- lifecycle ---------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.qs_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def state_bytes_per_env(self) -> int:
        return int(self.lib.qs_state_bytes_per_env(self._h))

    # -- env API -----------------------------------------------------------------------------------
    def reset(self, mask: torch.Tensor | None = None) -> torch.Tensor:
        """Reset all envs (mask None) or the masked ones; returns the obs buffer f32[n, obs_dim]."""
        mp = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mp = C.c_void_p(mask.data_ptr())
        check(self.lib, self._h, self.lib.qs_reset(self._h, mp, C.c_void_p(self.obs.data_ptr()), self._stream()), "qs_reset")
        return self.obs

    def step(self, actions: torch.Tensor) -> StepOut:
        """actions f32[n,4] on this device (not clipped here: SB3 clips before env.step)."""
        if actions.dtype != torch.float32 or actions.device != self.device or tuple(actions.shape) != (self.n_envs, 4):
            raise ValueError(f"actions must be float32[{self.n_envs},4] on {self.device}")
        if not actions.is_contiguous():
            actions = actions.contiguous()
        p = lambda t: C.c_void_p(t.data_ptr())
        check(self.lib, self._h,
              self.lib.qs_step(self._h, p(actions), p(self.obs), p(self.reward), p(self.flags), p(self.terminal_obs),
                               p(self.ep_return), p(self.ep_len), self._stream()), "qs_step")
        return StepOut(self.obs, self.reward, self.flags, self.terminal_obs, self.ep_return, self.ep_len)

    def step_many(self, T: int, actions: torch.Tensor | None = None, action_seed: int = 0, store_actions: bool = False,
                  obs_last_only: bool = False, store_terminal: bool = False, update_obs: bool = True) -> dict:
        """T steps in ONE kernel launch (`qs_step_many`): the hidden state stays in registers across the steps.  `actions`
        f32[T,n,4] time-major, or None: uniform-random actions over the action box drawn in the kernel (Philox on `action_seed`,
        the global env id and a device-resident step counter, so repeated calls and CUDA-graph replays draw fresh actions).
        Returns time-major device tensors {"obs": [T,n,D] (or [n,D] with obs_last_only), "reward": [T,n], "flags": [T,n], and
        "actions" / "terminal_obs" / "ep_return" / "ep_len" when requested}; the buffers are reused by the next call with the
        same T.  `self.obs` holds the observations after the last step (unless update_obs=False).  RK4 handles only."""
        n, d, dev = self.n_envs, self.obs_dim, self.device
        key = (int(T), bool(store_actions), bool(obs_last_only), bool(store_terminal))
        buf = getattr(self, "_many", None)
        if buf is None or buf["key"] != key:
            buf = {"key": key, "obs": self.obs if obs_last_only else torch.empty((T, n, d), dtype=torch.float32, device=dev),
                   "reward": torch.empty((T, n), dtype=self.real_dtype, device=dev), "flags": torch.zeros((T, n), dtype=torch.uint8, device=dev)}
            if store_actions:
                buf["actions"] = torch.empty((T, n, 4), dtype=torch.float32, device=dev)
            if store_terminal:
                buf["terminal_obs"] = torch.zeros((T, n, d), dtype=torch.float32, device=dev)
                buf["ep_return"] = torch.zeros((T, n), dtype=self.real_dtype, device=dev)
                buf["ep_len"] = torch.zeros((T, n), dtype=torch.int32, device=dev)
            self._many = buf
            if not hasattr(self, "_action_step"):
                self._action_step = torch.zeros(1, dtype=torch.int64, device=dev)
        a = _cabi.QsStepManyArgs()
        p = lambda t: t.data_ptr() if t is not None else None
        a.T, a.obs_last_only = int(T), int(bool(obs_last_only))
        if actions is not None:
            if actions.dtype != torch.float32 or tuple(actions.shape) != (T, n, 4) or not actions.is_contiguous() or actions.device != dev:
                raise ValueError(f"actions must be contiguous float32[{T},{n},4] on {dev}")
            a.actions = p(actions)
        a.action_seed = int(action_seed) & 0xFFFFFFFFFFFFFFFF
        a.action_step = p(self._action_step)
        a.action_lo[:] = (0.0, -1.0, -1.0, -1.0)          # the env's action box (rl_env_scaledObs.py:20-24)
        a.action_hi[:] = (2.0, 1.0, 1.0, 1.0)
        a.actions_out = p(buf.get("actions"))
        a.obs_out, a.reward_out, a.flags_out = p(buf["obs"]), p(buf["reward"]), p(buf["flags"])
        a.terminal_obs_out, a.ep_return_out, a.ep_len_out = p(buf.get("terminal_obs")), p(buf.get("ep_return")), p(buf.get("ep_len"))
        check(self.lib, self._h, self.lib.qs_step_many(self._h, C.byref(a), self._stream()), "qs_step_many")
        if not obs_last_only and update_obs:                  # keep `self.obs` = the observations after the last step (one D2D copy)
            self.obs.copy_(buf["obs"][T - 1])
        return {k: v for k, v in buf.items() if k != "key"}

    def step_range(self, first: int, count: int, actions: torch.Tensor, stream: torch.cuda.Stream | None = None) -> None:
        """Step envs [first, first + count) only (first a multiple of 32); `actions` is the f32[count,4] slice for them.  Results
        land in the same rows of the persistent output buffers.  Ordered on `stream` (default: the current stream) -- sub-ranges
        on different streams run independently, which is what QuadVecEnv's chunked host pipeline uses."""
        if actions.dtype != torch.float32 or tuple(actions.shape) != (count, 4) or not actions.is_contiguous():
            raise ValueError(f"actions must be contiguous float32[{count},4]")
        sl = slice(first, first + count)
        p = lambda t: C.c_void_p(t[sl].data_ptr())
        st = C.c_void_p((stream or torch.cuda.current_stream(self.device)).cuda_stream)
        check(self.lib, self._h,
              self.lib.qs_step_range(self._h, first, count, C.c_void_p(actions.data_ptr()), p(self.obs), p(self.reward), p(self.flags),
                                     p(self.terminal_obs), p(self.ep_return), p(self.ep_len), st), "qs_step_range")

    def fuse_obs_moments(self, moments: torch.Tensor | None, shift_stats: torch.Tensor | None = None,
                         merge_stats: torch.Tensor | None = None, exchange=None) -> None:
        """From now on every step() also writes (n, mean[D], M2[D]) of the returned observations into `moments` (f64[1+2D]):
        the batch statistics VecNormalize needs, reduced inside the step kernel.  None switches it off.
        The kernel centres its sums on the mean already in `moments` (when its count is > 0), so seed it with the statistics
        of the current observations (DeviceRunningMeanStd.attach does) to keep near-constant columns well conditioned."""
        if moments is not None:
            assert moments.dtype == torch.float64 and moments.numel() == 1 + 2 * self.obs_dim and moments.device == self.device
            assert shift_stats is None or (shift_stats.dtype == torch.float64 and shift_stats.numel() == 1 + 2 * self.obs_dim)
        self._mom_keep = (moments, shift_stats, merge_stats)
        check(self.lib, self._h, self.lib.qs_step_moments(self._h, C.c_void_p(moments.data_ptr()) if moments is not None else None,
                                                          C.c_void_p(shift_stats.data_ptr()) if shift_stats is not None else None), "qs_step_moments")
        # merge_stats (f64[1+2D] running count/mean/var): every step() also performs RunningMeanStd.update on it (single GPU)
        # exchange (a connected qs_xchg handle, several ranks): the kernel that finishes the moments also exchanges them with the peers
        # and merges every rank's triplet into merge_stats (qs_step_moments_exchange)
        if moments is not None:
            assert merge_stats is None or (merge_stats.dtype == torch.float64 and merge_stats.numel() == 1 + 2 * self.obs_dim)
            if exchange is not None:
                assert merge_stats is not None
                check(self.lib, self._h, self.lib.qs_step_moments_merge(self._h, None), "qs_step_moments_merge")
                check(self.lib, self._h, self.lib.qs_step_moments_exchange(self._h, exchange, C.c_void_p(merge_stats.data_ptr())),
                      "qs_step_moments_exchange")
            else:
                check(self.lib, self._h, self.lib.qs_step_moments_exchange(self._h, None, None), "qs_step_moments_exchange")
                check(self.lib, self._h, self.lib.qs_step_moments_merge(self._h, C.c_void_p(merge_stats.data_ptr()) if merge_stats is not None else None),
                      "qs_step_moments_merge")

    # -- state injection / extraction (parity tests, plotting façade) ------------------------------
    def get_state(self, fields=None) -> dict[str, torch.Tensor]:
        fields = list(fields or _STATE_FIELDS)
        out, view = {}, QsStateView()
        for name in fields:
            dt, shp = _STATE_FIELDS[name]
            out[name] = torch.empty((self.n_envs, *shp), dtype=dt, device=self.device)
            setattr(view, name, out[name].data_ptr())
        check(self.lib, self._h, self.lib.qs_get_state(self._h, C.byref(view), self._stream()), "qs_get_state")
        return out

    def set_state(self, **fields) -> None:
        view, keep = QsStateView(), []
        for name, val in fields.items():
            dt, shp = _STATE_FIELDS[name]
            t = torch.as_tensor(val).to(device=self.device, dtype=dt).contiguous()
            if tuple(t.shape) != (self.n_envs, *shp):
                raise ValueError(f"{name}: expected shape {(self.n_envs, *shp)}, got {tuple(t.shape)}")
            keep.append(t)
            setattr(view, name, t.data_ptr())
        check(self.lib, self._h, self.lib.qs_set_state(self._h, C.byref(view), self._stream()), "qs_set_state")
        torch.cuda.current_stream(self.device).synchronize()  # `keep` must outlive the kernel

    def reset_uniforms(self, env_ids: torch.Tensor, episodes: torch.Tensor) -> torch.Tensor:
        """The RESET_UNIFORMS unit uniforms the reset of (global env id, episode) may consume -- test hook."""
        env_ids = env_ids.to(device=self.device, dtype=torch.int64).contiguous()
        episodes = episodes.to(device=self.device, dtype=torch.int32).contiguous()
        out = torch.empty((env_ids.numel(), _cabi.RESET_UNIFORMS), dtype=torch.float64, device=self.device)
        check(self.lib, self._h, self.lib.qs_reset_uniforms(self._h, C.c_void_p(env_ids.data_ptr()), C.c_void_p(episodes.data_ptr()),
                                                           env_ids.numel(), C.c_void_p(out.data_ptr()), self._stream()), "qs_reset_uniforms")
        return out

    # -- dynamics randomisation ------------------------------------------------------------------
    def randomize_dynamics(self, cfg: dict | None) -> None:
        """Arm (dict with keys mass, inertia, thrust, wind and optional seed, default the env seed) or disarm (None) dynamics
        randomisation.  Arming draws every env's parameters for its current episode; every later reset draws its episode's."""
        if cfg is None:
            check(self.lib, self._h, self.lib.qs_dynamics_randomization(self._h, None, self._stream()), "qs_dynamics_randomization")
            self.dynamics_randomization = None
            return
        unknown = set(cfg) - {"mass", "inertia", "thrust", "wind", "seed"}
        if unknown:
            raise ValueError(f"dynamics_randomization: unknown keys {sorted(unknown)} (mass, inertia, thrust, wind, seed)")
        r = _cabi.QsDynamicsRand()
        r.seed = int(cfg.get("seed", self.seed)) & 0xFFFFFFFFFFFFFFFF
        r.mass_rel, r.inertia_rel = float(cfg.get("mass", 0.0)), float(cfg.get("inertia", 0.0))
        r.thrust_rel, r.wind = float(cfg.get("thrust", 0.0)), float(cfg.get("wind", 0.0))
        check(self.lib, self._h, self.lib.qs_dynamics_randomization(self._h, C.byref(r), self._stream()), "qs_dynamics_randomization")
        self.dynamics_randomization = dict(cfg)

    def _dyn_rows(self) -> torch.Tensor:
        out = torch.empty((self.n_envs, _cabi.DYN_PARAMS), dtype=torch.float64, device=self.device)
        check(self.lib, self._h, self.lib.qs_get_dynamics(self._h, C.c_void_p(out.data_ptr()), self._stream()), "qs_get_dynamics")
        return out

    def dynamics(self) -> dict[str, torch.Tensor]:
        """The current episode's parameters of every env (float64 device tensors): mass_scale [n], inertia_scale [n],
        thrust_scale [n,4], wind [n,3] (N, world frame)."""
        d = self._dyn_rows()
        return {"mass_scale": d[:, 0].clone(), "inertia_scale": d[:, 1].clone(), "thrust_scale": d[:, 2:6].clone(),
                "wind": d[:, 6:9].clone()}

    def set_dynamics(self, mass_scale=None, inertia_scale=None, thrust_scale=None, wind=None) -> None:
        """Overwrite the parameters of every env (fields left None keep their values) until that env's next reset.  Scalars
        broadcast.  Needs armed randomisation; mass_scale and inertia_scale must be > 0, thrust_scale >= 0, all finite."""
        d = self._dyn_rows()
        n = self.n_envs
        for name, val, cols, shape in (("mass_scale", mass_scale, slice(0, 1), (n,)), ("inertia_scale", inertia_scale, slice(1, 2), (n,)),
                                       ("thrust_scale", thrust_scale, slice(2, 6), (n, 4)), ("wind", wind, slice(6, 9), (n, 3))):
            if val is None:
                continue
            t = torch.as_tensor(val, dtype=torch.float64, device=self.device)
            try:
                t = torch.broadcast_to(t, shape)
            except RuntimeError:
                raise ValueError(f"{name}: expected shape {shape} (or broadcastable), got {tuple(t.shape)}") from None
            if not bool(torch.isfinite(t).all()):
                raise ValueError(f"{name}: values must be finite")
            if name in ("mass_scale", "inertia_scale") and not bool((t > 0).all()):
                raise ValueError(f"{name}: values must be > 0")
            if name == "thrust_scale" and not bool((t >= 0).all()):
                raise ValueError(f"{name}: values must be >= 0")
            d[:, cols] = t.reshape(n, -1)
        check(self.lib, self._h, self.lib.qs_set_dynamics(self._h, C.c_void_p(d.data_ptr()), self._stream()), "qs_set_dynamics")
        torch.cuda.current_stream(self.device).synchronize()  # `d` must outlive the kernel

    def lsoda_stats(self):
        """(i32[n,4] = nst, nfe, nqu, status ; f64[n,2] = hu, tcur) of the last step in LSODA mode."""
        cnt = torch.empty((self.n_envs, 4), dtype=torch.int32, device=self.device)
        stp = torch.empty((self.n_envs, 2), dtype=torch.float64, device=self.device)
        check(self.lib, self._h, self.lib.qs_lsoda_stats(self._h, C.c_void_p(cnt.data_ptr()), C.c_void_p(stp.data_ptr()), self._stream()),
              "qs_lsoda_stats")
        return cnt, stp
