"""QuadVecEnv -- the Stable-Baselines3 `VecEnv` surface over the B200 batched simulator.

Drop-in for what the reference builds with
    env = make_vec_env(WaypointQuadEnv, n_envs=8)            (initial-implementation-v1/rl_train_vecN.py:10,
                                                               initial-implementation-v2/rl_train.py:24)
i.e. `DummyVecEnv([Monitor(WaypointQuadEnv()) ...])`: NumPy in, NumPy out, auto-reset with
`info["terminal_observation"]`, `info["TimeLimit.truncated"]`, Monitor-style `info["episode"]`, plus the
reference env's own info keys (`success`, `stopped`, `crashed`, `out_of_bounds`).

SB3 protocol restated from stable_baselines3 2.6.0 `common/vec_env/{base_vec_env,dummy_vec_env}.py` and
`common/monitor.py` (SB3 is not installable in this image; when it is importable QuadVecEnv subclasses
`stable_baselines3.common.vec_env.VecEnv` so PPO / VecNormalize / evaluate_policy accept it).

Host<->device traffic per step is exactly: actions f32[n,4] up; obs f32[n,D], reward, flags down, through
pinned staging buffers on the env's stream.  `infos` dictionaries are built only for envs that finished
or reported an info key; all other entries are one shared empty dict (at 1M envs a per-env dict would cost
more than the step).  The zero-copy path is BatchedQuadEnv.
"""
from __future__ import annotations

import os
import time
from typing import Any, Sequence

import numpy as np
import torch

from . import _cabi
from .batched_env import BatchedQuadEnv

try:  # pragma: no cover - SB3 is absent in the build image
    from stable_baselines3.common.vec_env import VecEnv as _SB3VecEnv
except Exception:  # noqa: BLE001
    _SB3VecEnv = object

try:  # pragma: no cover
    from gymnasium import spaces as _spaces
except Exception:  # noqa: BLE001
    _spaces = None


class Box:
    """Minimal stand-in for gymnasium.spaces.Box when gymnasium is not installed."""

    def __init__(self, low, high, shape=None, dtype=np.float32):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(shape if shape is not None else np.shape(low))
        self.low = np.broadcast_to(np.asarray(low, dtype=self.dtype), self.shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=self.dtype), self.shape).copy()

    def sample(self):
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return np.random.uniform(lo, hi).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))


def _box(low, high, shape=None, dtype=np.float32):
    if _spaces is not None:
        return _spaces.Box(low=np.asarray(low, dtype=dtype) if shape is None else low, high=np.asarray(high, dtype=dtype) if shape is None else high,
                           shape=shape, dtype=dtype)
    return Box(low, high, shape, dtype)


_EMPTY: dict = {}


class LazyInfos:
    """Sequence of per-env info dicts that are only materialised when indexed (`info_mode="lazy"`).

    `done_indices` lists the envs that finished this step; indexing any other env that raised no info key
    returns the shared empty dict, so a consumer that only looks at finished envs does O(#done) work."""

    def __init__(self, env: "QuadVecEnv", flags: np.ndarray, dones: np.ndarray):
        self._env, self._flags, self._dones = env, flags.copy(), dones
        self.done_indices = np.nonzero(dones)[0]
        self._cache: dict[int, dict] = {}
        self._fetched = None

    def __len__(self):
        return self._flags.shape[0]

    def _fetch(self):
        if self._fetched is None:
            self._fetched = self._env._fetch_done(self.done_indices)
        return self._fetched

    def __getitem__(self, i):
        i = int(i)
        f = int(self._flags[i])
        if f == 0:
            return _EMPTY
        if i not in self._cache:
            extra = None
            if self._dones[i]:
                tobs, ep_r, ep_l, t_now = self._fetch()
                k = int(np.searchsorted(self.done_indices, i))
                extra = (tobs[k], ep_r[k], ep_l[k], t_now)
            self._cache[i] = self._env._make_info(f, extra)
        return self._cache[i]

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class QuadVecEnv(_SB3VecEnv):
    """VecEnv of `num_envs` WaypointQuadEnv instances living on one B200."""

    metadata = {"render_modes": []}

    def __init__(self, num_envs: int = 8, env_version: int = 2, precision: str = "f32", integrator: str = "rk4",
                 substeps: int = 1, obs_scaled: bool = True, device: int | None = None, seed: int = 0,
                 env_id_offset: int = 0, monitor: bool = True, info_mode: str = "dict", v2_random_waypoints: bool = False,
                 pipeline_chunks: int | None = None, dynamics_randomization: dict | None = None):
        """pipeline_chunks: split a step into this many env sub-ranges, each on its own stream -- actions of chunk c+1 are copied
        up while chunk c steps and its observations come down, so the PCIe link works in both directions at once.
        None: 4 from 262,144 envs, else 1.  dynamics_randomization: see BatchedQuadEnv."""
        self.sim = BatchedQuadEnv(num_envs, env_version=env_version, precision=precision, integrator=integrator,
                                  substeps=substeps, obs_scaled=obs_scaled, auto_reset=True, device=device,
                                  env_id_offset=env_id_offset, seed=seed, v2_random_waypoints=v2_random_waypoints,
                                  dynamics_randomization=dynamics_randomization)
        d = self.sim.obs_dim
        observation_space = _box(-np.inf, np.inf, (d,), np.float32)      # rl_env_scaledObs.py:14-17
        action_space = _box(np.array([0, -1, -1, -1], dtype=np.float32), np.array([2.0, 1, 1, 1], dtype=np.float32))  # :20-24
        if _SB3VecEnv is not object:
            super().__init__(num_envs, observation_space, action_space)
        else:
            self.num_envs, self.observation_space, self.action_space = num_envs, observation_space, action_space
            self.render_mode = None
            self.reset_infos = [{} for _ in range(num_envs)]
        self.monitor = monitor
        if info_mode not in ("dict", "lazy"):
            raise ValueError("info_mode must be 'dict' (SB3 list of dicts) or 'lazy'")
        self.info_mode = info_mode
        self._t_start = time.time()
        self._stream = torch.cuda.Stream(device=self.sim.device)
        pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
        n = num_envs
        self._h_actions = pin((n, 4), torch.float32)
        self._d_actions = torch.empty((n, 4), dtype=torch.float32, device=self.sim.device)
        # two sets of pinned result buffers, used alternately: the arrays returned by step_wait() are views
        # of one set and stay valid until the step after next (no per-step host memcpy of n*D floats)
        self._h_bufs = [(pin((n, d), torch.float32), pin((n,), self.sim.real_dtype), pin((n,), torch.uint8)) for _ in range(2)]
        self._flip = 0
        self._h_obs, self._h_reward, self._h_flags = self._h_bufs[0]
        self._pending = False
        self._transform = None      # optional device-side post-processing of a step (QuadVecNormalize installs one)
        if pipeline_chunks is None:
            pipeline_chunks = int(os.environ.get("QS_PIPELINE_CHUNKS", "4")) if (n >= 262144 and integrator == "rk4") else 1
        self._chunks = []           # (first, count) sub-ranges of whole warp tiles
        if pipeline_chunks > 1:
            per = ((n + pipeline_chunks - 1) // pipeline_chunks + 31) // 32 * 32
            self._chunks = [(f, min(per, n - f)) for f in range(0, n, per)]
            self._chunk_streams = [torch.cuda.Stream(device=self.sim.device) for _ in self._chunks]
        self.h2d_bytes_per_step = n * 4 * 4
        self.d2h_bytes_per_step = n * d * 4 + n * self._h_reward.element_size() + n

    # ---- VecEnv protocol -------------------------------------------------------------------------
    def reset(self) -> np.ndarray:
        with torch.cuda.stream(self._stream):
            obs = self.sim.reset()
            self._h_obs.copy_(obs, non_blocking=True)
        self._stream.synchronize()
        self.reset_infos = [{} for _ in range(self.num_envs)]
        return self._h_obs.numpy().copy()

    @property
    def pipelined(self) -> bool:
        """True when step() goes through in chunks on separate streams (qs_step_range).  A device-side transform that needs the
        WHOLE batch before it can produce any output row -- QuadVecNormalize updates the running statistics from all observations
        of the step and only then normalises them -- switches the host pipeline off: one launch, one upload, one download."""
        return len(self._chunks) > 1 and self._transform is None

    def step_async(self, actions: np.ndarray) -> None:
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.num_envs, 4)
        src = torch.from_numpy(a)
        if not src.is_pinned():            # stage through pinned memory unless the caller already handed us a pinned array
            self._h_actions.numpy()[...] = a
            src = self._h_actions
        self._flip ^= 1
        self._h_obs, self._h_reward, self._h_flags = self._h_bufs[self._flip]
        if self.pipelined:
            sim = self.sim
            for (f, c), st in zip(self._chunks, self._chunk_streams):
                sl = slice(f, f + c)
                with torch.cuda.stream(st):
                    self._d_actions[sl].copy_(src[sl], non_blocking=True)
                    sim.step_range(f, c, self._d_actions[sl], st)
                    self._h_obs[sl].copy_(sim.obs[sl], non_blocking=True)
                    self._h_reward[sl].copy_(sim.reward[sl], non_blocking=True)
                    self._h_flags[sl].copy_(sim.flags[sl], non_blocking=True)
            self._pending = True
            return
        with torch.cuda.stream(self._stream):
            self._d_actions.copy_(src, non_blocking=True)
            out = self.sim.step(self._d_actions)
            obs_t, rew_t = self._transform(out) if self._transform is not None else (out.obs, out.reward)
            self._h_obs.copy_(obs_t, non_blocking=True)
            self._h_reward.copy_(rew_t, non_blocking=True)
            self._h_flags.copy_(out.flags, non_blocking=True)
        self._pending = True

    def step_wait(self):
        assert self._pending, "step_wait() without step_async()"
        if self.pipelined:
            for st in self._chunk_streams:
                st.synchronize()
        self._stream.synchronize()
        self._pending = False
        obs = self._h_obs.numpy()
        rewards = self._h_reward.numpy() if self._h_reward.dtype == torch.float32 else self._h_reward.numpy().astype(np.float32)
        flags = self._h_flags.numpy()
        dones = (flags & 3) != 0
        infos = self._build_infos(flags, dones)
        return obs, rewards, dones, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def _fetch_done(self, done_ids: np.ndarray):
        """terminal_observation / Monitor stats of the finished envs, gathered on the device first."""
        if done_ids.size == 0:
            d = self.sim.obs_dim
            return np.zeros((0, d), np.float32), np.zeros(0), np.zeros(0, np.int32), 0.0
        idx = torch.from_numpy(done_ids).to(self.sim.device)
        with torch.cuda.stream(self._stream):
            tobs = self.sim.terminal_obs.index_select(0, idx).cpu().numpy()
            ep_r = self.sim.ep_return.index_select(0, idx).cpu().numpy()
            ep_l = self.sim.ep_len.index_select(0, idx).cpu().numpy()
        return tobs, ep_r, ep_l, round(time.time() - self._t_start, 6)

    def _make_info(self, f: int, extra) -> dict:
        info: dict[str, Any] = {}
        if f & _cabi.FLAG_SUCCESS:                       # {'success': True, 'stopped': ...}
            info["success"] = True
            info["stopped"] = bool(f & _cabi.FLAG_STOPPED)
        elif f & _cabi.FLAG_CRASHED:                     # {'success': False, 'crashed': True}
            info["success"] = False
            info["crashed"] = True
        elif f & _cabi.FLAG_OOB:                         # {'success': False, 'out_of_bounds': True}
            info["success"] = False
            info["out_of_bounds"] = True
        if extra is not None:                            # DummyVecEnv + Monitor additions for a finished env
            tobs, ep_r, ep_l, t_now = extra
            term, trunc = bool(f & _cabi.FLAG_TERMINATED), bool(f & _cabi.FLAG_TRUNCATED)
            info["TimeLimit.truncated"] = trunc and not term
            info["terminal_observation"] = tobs
            if self.monitor:
                info["episode"] = {"r": round(float(ep_r), 6), "l": int(ep_l), "t": t_now}
        return info

    def _build_infos(self, flags: np.ndarray, dones: np.ndarray):
        if self.info_mode == "lazy":
            return LazyInfos(self, flags, dones)
        infos: list[dict] = [_EMPTY] * self.num_envs
        interesting = np.nonzero(flags != 0)[0]
        if interesting.size == 0:
            return infos
        done_ids = interesting[dones[interesting]]
        tobs, ep_r, ep_l, t_now = self._fetch_done(done_ids)
        k = 0
        for i in interesting:
            extra = None
            if dones[i]:
                extra = (tobs[k], ep_r[k], ep_l[k], t_now)
                k += 1
            infos[i] = self._make_info(int(flags[i]), extra)
        return infos

    def close(self) -> None:
        self.sim.close()

    # ---- the rest of the abstract surface ---------------------------------------------------------
    def get_attr(self, attr_name: str, indices=None) -> list:
        ids = self._indices(indices)
        if attr_name in ("waypoint_list", "current_waypoint", "waypoint_index", "state", "final_yaw", "current_step"):
            st = {k: v.cpu().numpy() for k, v in self.sim.get_state().items()}
            out = []
            for i in ids:
                nwp = int(st["n_wp"][i])
                wl = [st["wp_list"][i, j].copy() for j in range(nwp)]
                val = {"waypoint_list": wl, "current_waypoint": wl[min(int(st["wp_index"][i]), nwp - 1)],
                       "waypoint_index": int(st["wp_index"][i]), "state": st["y"][i].copy(),
                       "final_yaw": float(st["final_yaw"][i]), "current_step": int(st["current_step"][i])}[attr_name]
                out.append(val)
            return out
        if attr_name == "render_mode":
            return [None for _ in ids]
        if attr_name == "dt":
            return [1.0 / 200.0 for _ in ids]
        raise AttributeError(f"QuadVecEnv has no per-env attribute {attr_name!r}")

    def set_attr(self, attr_name: str, value, indices=None) -> None:
        raise NotImplementedError("per-env attributes live on the GPU; use sim.set_state(...)")

    def env_method(self, method_name: str, *args, indices=None, **kwargs) -> list:
        raise NotImplementedError(f"env_method({method_name!r}) is not available on the batched GPU env")

    def env_is_wrapped(self, wrapper_class, indices=None) -> list[bool]:
        return [False for _ in self._indices(indices)]

    def seed(self, seed: int | None = None) -> Sequence[None | int]:
        # like the reference, whose reset(seed) never reaches np.random (rl_env_scaledObs.py:40-44), the
        # episode stream is fixed at construction (Philox key); report it back
        return [self.sim.cfg.seed for _ in range(self.num_envs)]

    def get_images(self):
        return [None] * self.num_envs

    def render(self, mode=None):
        return None

    def _indices(self, indices):
        if indices is None:
            return range(self.num_envs)
        if isinstance(indices, int):
            return [indices]
        return list(indices)
