"""PopulationPPO -- K independent QuadPPO agents (seeds and hyper-parameters) trained in the same kernel launches on one GPU.

What a seed study or a hyper-parameter sweep of the reference runs as K separate `PPO("MlpPolicy", env, ...).learn()` processes
(its authors tried ent_coef 0.01 / 0.0005 / 0.0001 and n_epochs 10 / 12 over continuation runs) as ONE training loop: agent a
owns envs [a*n, (a+1)*n) of one BatchedQuadEnv(K*n, ...) and trains bit for bit like the solo run
    QuadPPO(BatchedQuadEnv(n, <same env kwargs>, env_id_offset=a*n), policy_impl="fp32", seed=seeds[a], <hyper of agent a>)
(parameters, Adam state, rollout buffers, env state, training statistics; ep_rew_mean up to the float64 summation order).

  * collection: K `normal_` draws (one generator per agent) into row blocks of one noise buffer, ONE population policy forward
    (`qs_policy_forward_pop`: each row is the fp32 FFMA kernel's row with its agent's blob), the env step of all K*n envs, the
    column-wise rollout-record kernels of QuadPPO, one step captured as a CUDA graph and replayed;
  * GAE over the whole [T, K*n] buffers (column-wise, so every column is its solo value);
  * update: per epoch one permutation per agent (its own generator, the solo's call order), translated to rows of the shared
    buffers; then ONE `qs_ppo_pop_update` launch per minibatch serves all K agents (per agent the solo kernel's CTAs, tiling and
    reduction order).
Per agent: seed, learning_rate, ent_coef, clip_range, vf_coef, max_grad_norm, normalize_advantage (qs_ppo_hyper), optionally an
initial state_dict.  Shared: n_steps, batch_size, n_epochs, gamma, gae_lambda and the env configuration.  No VecNormalize, one
rank (DESIGN section 13).
"""
from __future__ import annotations

import ctypes as C
import warnings

import numpy as np
import torch
import torch.distributed as dist

from . import sb3_compat
from ._cabi import QsPpoHyper, load_library
from .policy import ACTION_HIGH, ACTION_LOW, NACT, pack_params, unpack_params
from .ppo import STAT_KEYS, QuadPPO, _bind, gae, init_state_dict

PER_AGENT = ("learning_rate", "ent_coef", "clip_range", "vf_coef", "max_grad_norm", "normalize_advantage")
DEFAULTS = {"learning_rate": 2e-4, "ent_coef": 0.01, "clip_range": 0.2, "vf_coef": 0.5, "max_grad_norm": 0.5, "normalize_advantage": True}
MAX_ENVS = 65536          # the time-limit bootstrap runs the critic on every env's terminal observation, as QuadPPO does up to here


def flat_rows(perms: torch.Tensor, n: int, K: int) -> torch.Tensor:
    """perms int64[K, T*n]: agent a's permutation of the rows of its own flat [T*n] buffers -> the same rows of the shared flat
    [T*K*n] buffers (time-major [T, K*n], agent a in columns [a*n, (a+1)*n)): (r // n) * K*n + a*n + r % n."""
    a = torch.arange(K, dtype=perms.dtype, device=perms.device).unsqueeze(1)
    return (perms // n) * (K * n) + a * n + perms % n


class PopulationPPO:
    def __init__(self, env, K: int, seeds, hyper: dict | None = None, n_steps: int = 64, batch_size: int = 65536, n_epochs: int = 10,
                 gamma: float = 0.995, gae_lambda: float = 0.9, state_dicts=None, rollout_graph: bool | None = None, vecnorm=None):
        K = int(K)
        if vecnorm is not None:
            raise ValueError("PopulationPPO does not support VecNormalize (its statistics span the whole env batch, not one agent)")
        if dist.is_initialized() and dist.get_world_size() > 1:
            raise ValueError("PopulationPPO is single-rank only")
        if K < 1 or env.n_envs % K != 0:
            raise ValueError(f"env.n_envs = {env.n_envs} is not K * n envs for K = {K}")
        if env.n_envs > MAX_ENVS:
            raise ValueError(f"K * n = {env.n_envs} envs; PopulationPPO supports at most {MAX_ENVS}")
        if int(n_steps) < 1:
            raise ValueError(f"n_steps must be >= 1, got {n_steps}")
        seeds = [int(s) for s in seeds]
        if len(seeds) != K:
            raise ValueError(f"{len(seeds)} seeds for K = {K} agents")
        hyper = dict(hyper or {})
        unknown = set(hyper) - set(PER_AGENT)
        if unknown:
            raise ValueError(f"hyper: unknown keys {sorted(unknown)} (per-agent keys: {', '.join(PER_AGENT)})")
        self.hyper = {k: self._per_agent(k, hyper.get(k, DEFAULTS[k]), K) for k in PER_AGENT}
        if state_dicts is not None and len(state_dicts) != K:
            raise ValueError(f"{len(state_dicts)} state_dicts for K = {K} agents")
        self.env, self.K, self.n, self.seeds = env, K, env.n_envs // K, seeds
        self.n_steps, self.batch_size, self.n_epochs = int(n_steps), int(batch_size), int(n_epochs)
        self.gamma, self.gae_lambda = gamma, gae_lambda
        dev, N, d, T = env.device, env.n_envs, env.obs_dim, self.n_steps
        self.device, self.obs_dim = dev, d
        self.lib = load_library()
        _bind(self.lib)
        sds = [state_dicts[a] if state_dicts is not None and state_dicts[a] is not None else init_state_dict(d, seeds[a]) for a in range(K)]
        blobs = [pack_params({k: np.asarray(v, dtype=np.float32) for k, v in sd.items()}, d) for sd in sds]
        self.params = torch.from_numpy(np.stack(blobs)).to(dev)                   # [K, n_params]: agent a's policy blob
        h = C.c_void_p()
        self._check(self.lib.qs_ppo_pop_create(dev.index or 0, d, K, C.byref(h)), "qs_ppo_pop_create")
        self._h = h
        self.gens = [torch.Generator(device=dev).manual_seed(s) for s in seeds]
        f32 = dict(dtype=torch.float32, device=dev)
        self.obs = torch.empty((T, N, d), **f32)
        self.actions = torch.empty((T, N, NACT), **f32)
        self.values, self.logp, self.rewards = torch.empty((T, N), **f32), torch.empty((T, N), **f32), torch.empty((T, N), **f32)
        self.advantages, self.returns = torch.empty((T, N), **f32), torch.empty((T, N), **f32)
        self.episode_starts = torch.zeros((T, N), dtype=torch.uint8, device=dev)
        self._noise = torch.empty((N, NACT), **f32)
        # policy outputs of the rollout forward, and of the critic-only forwards (terminal observations, last values)
        self._pol = (torch.empty((N, NACT), **f32), torch.empty((N, NACT), **f32), torch.empty(N, **f32), torch.empty(N, **f32))
        self._aux = (torch.empty((N, NACT), **f32), torch.empty((N, NACT), **f32), torch.empty(N, **f32), torch.empty(N, **f32))
        self._lo, self._hi = (C.c_float * 4)(*ACTION_LOW), (C.c_float * 4)(*ACTION_HIGH)
        self._last_dones = torch.ones(N, dtype=torch.uint8, device=dev)
        self._last_obs = None
        self._use_graph = True if rollout_graph is None else bool(rollout_graph)
        self._graph = None
        self._t = torch.zeros(1, dtype=torch.int64, device=dev)
        self._rec_ws = torch.zeros(2 * 1024 + 1, dtype=torch.float64, device=dev)   # qs_rollout_record_post workspace
        self._rec_stats = torch.zeros(2, dtype=torch.float64, device=dev)        # its whole-batch episode sums: not used
        self._ep_stats = torch.zeros((K, 2), dtype=torch.float64, device=dev)    # per agent: sum of finished returns, count
        self._zero = torch.zeros((), dtype=torch.float64, device=dev)
        self._stats = torch.zeros((K, len(STAT_KEYS)), **f32)
        self.num_timesteps, self._n_updates = 0, 0
        self.ep_rew_mean, self.ep_count = [float("nan")] * K, [0] * K

    @staticmethod
    def _per_agent(key, value, K):
        vals = list(value) if isinstance(value, (list, tuple, np.ndarray)) else [value] * K
        if len(vals) != K:
            raise ValueError(f"hyper[{key!r}] has {len(vals)} values for K = {K} agents")
        return [bool(v) for v in vals] if key == "normalize_advantage" else [float(v) for v in vals]

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {self.lib.qs_ppo_last_error().decode()}")

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- rollout -------------------------------------------------------------------------------------
    def _forward(self, obs, noise, out):
        """All K agents' policy forwards on their row blocks of obs [K*n, d] (qs_policy_forward_pop) into the buffers `out`."""
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        act, act_c, val, lp = out
        rc = self.lib.qs_policy_forward_pop(p(self.params), self.obs_dim, self.K, p(obs), p(noise), self.n, p(act), p(act_c),
                                            C.byref(self._lo), C.byref(self._hi), p(val), p(lp), self._stream())
        if rc != 0:
            raise RuntimeError(f"qs_policy_forward_pop failed ({rc}): {self.lib.qs_policy_last_error().decode()}")
        return out

    def _step(self):
        """One collection step of all agents with every address fixed (QuadPPO._graph_step_kernels on the whole batch, the noise
        drawn per agent, the episode statistics reduced per agent): capturable, and the body of the replayed graph."""
        env, lib, n, K = self.env, self.lib, self.n, self.K
        for a, g in enumerate(self.gens):
            self._noise[a * n:(a + 1) * n].normal_(generator=g)       # what the solo's normal_ on its own [n, 4] buffer draws
        raw = env.obs
        act, act_c, val, lp = self._forward(raw, self._noise, self._pol)
        p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None
        st = self._stream()
        N = env.n_envs
        rc = lib.qs_rollout_record_pre(p(self._t), N, self.obs_dim, p(raw), p(act), p(val), p(lp), p(self._last_dones), p(self.obs),
                                       p(self.actions), p(self.values), p(self.logp), p(self.episode_starts), st)
        if rc != 0:
            raise RuntimeError(f"qs_rollout_record_pre failed ({rc}): {lib.qs_gae_last_error().decode()}")
        out = env.step(act_c)
        tv = self._forward(out.terminal_obs, None, self._aux)[2]               # time-limit bootstrap: critic on every row
        rc = lib.qs_rollout_record_post(p(self._t), N, p(out.reward), int(out.reward.dtype == torch.float64), p(out.flags), p(out.ep_return),
                                        p(tv), float(self.gamma), None, 0.0, 0.0, p(self.rewards), p(self._last_dones), p(self._rec_stats),
                                        p(self._rec_ws), st)
        if rc != 0:
            raise RuntimeError(f"qs_rollout_record_post failed ({rc}): {lib.qs_gae_last_error().decode()}")
        done = ((out.flags & 3) != 0).view(K, n)
        self._ep_stats[:, 0] += torch.where(done, out.ep_return.view(K, n).double(), self._zero).sum(1)
        self._ep_stats[:, 1] += done.sum(1)

    def _collect_graph(self) -> None:
        """As QuadPPO._collect_graph: the first two steps of the first collection run eagerly (lazy initialisation must not happen
        under capture), the third is captured with every agent's generator registered, the rest are replays."""
        env = self.env
        if self._graph is not None and self._graph[1] != float(self.gamma):
            self._graph = None                                   # the captured step has gamma baked in
        done = 0
        if self._graph is None:
            for _ in range(2):
                self._step()
            done = 2
            torch.cuda.synchronize(env.device)
            try:
                g = torch.cuda.CUDAGraph()
                for gen in self.gens:
                    g.register_generator_state(gen)
                with torch.cuda.graph(g):
                    self._step()
            except Exception as exc:  # noqa: BLE001 -- a launch-mode optimisation only: the same step body goes on eagerly
                warnings.warn(f"PopulationPPO: the collection step could not be captured as a CUDA graph ({exc}); collecting eagerly")
                torch.cuda.synchronize(env.device)
                self._use_graph = False
                for _ in range(done, self.n_steps):
                    self._step()
                return
            self._graph = (g, float(self.gamma))
        for _ in range(done, self.n_steps):
            self._graph[0].replay()

    def collect_rollouts(self):
        env = self.env
        if self._last_obs is None:
            self._last_obs = env.reset()
        self._ep_stats.zero_()
        self._t.zero_()
        if self._use_graph and self.n_steps >= 4 and self._last_obs.data_ptr() == env.obs.data_ptr():
            self._collect_graph()
        else:
            for _ in range(self.n_steps):
                self._step()
        self._last_obs = env.obs
        last_values = self._forward(env.obs, None, self._aux)[2]
        gae(self.rewards, self.values, self.episode_starts, last_values, self._last_dones, self.gamma, self.gae_lambda,
            out=(self.advantages, self.returns))
        self.num_timesteps += self.n_steps * self.n
        stats = self._ep_stats.tolist()
        self.ep_rew_mean = [s / c if c > 0 else float("nan") for s, c in stats]
        self.ep_count = [int(c) for _, c in stats]

    # ---- update --------------------------------------------------------------------------------------
    def _set_hyper(self):
        hp = self.hyper
        self._hp = (QsPpoHyper * self.K)(*[QsPpoHyper(hp["clip_range"][a], hp["ent_coef"][a], hp["vf_coef"][a], hp["max_grad_norm"][a],
                                                      hp["learning_rate"][a], 0.9, 0.999, 1e-5, int(hp["normalize_advantage"][a]), 0)
                                           for a in range(self.K)])
        self._check(self.lib.qs_ppo_pop_set_hyper(self._h, self._hp, self._stream()), "qs_ppo_pop_set_hyper")

    def train(self) -> list[dict]:
        """PPO.train of every agent: n_epochs passes in shuffled minibatches (the ragged last one included), ONE population-update
        launch per minibatch for all agents.  The hyper-parameters are read from self.hyper here, so they may change between
        iterations.  Returns each agent's statistics of its last minibatch."""
        self._set_hyper()
        T, N = self.rewards.shape
        n, K = self.n, self.K
        total = T * n
        flat = lambda x: x.reshape(T * N, *x.shape[2:])
        obs, act, oldlp, adv, ret = map(flat, (self.obs, self.actions, self.logp, self.advantages, self.returns))
        p = lambda t: C.c_void_p(t.data_ptr())
        bs = min(self.batch_size, total)
        st = self._stream()
        for _ in range(self.n_epochs):
            perms = torch.stack([torch.randperm(total, device=self.device, generator=g) for g in self.gens])
            rows = flat_rows(perms, n, K)
            for start in range(0, total, bs):
                self._check(self.lib.qs_ppo_pop_update(self._h, p(self.params), p(obs), p(act), p(oldlp), p(adv), p(ret),
                                                       C.c_void_p(rows.data_ptr() + 8 * start), total, min(bs, total - start),
                                                       p(self._stats), st), "qs_ppo_pop_update")
        self._n_updates += self.n_epochs
        return [dict(zip(STAT_KEYS, s)) for s in self._stats.tolist()]

    def learn(self, total_timesteps_per_agent: int, log=None):
        """Train until every agent has collected total_timesteps_per_agent steps.  log: called per iteration with one dict per
        agent (its statistics, `agent`, `timesteps`, `ep_rew_mean`, `episodes`)."""
        while self.num_timesteps < total_timesteps_per_agent:
            self.collect_rollouts()
            infos = self.train()
            if log:
                for a, info in enumerate(infos):
                    log(dict(info, agent=a, timesteps=self.num_timesteps, ep_rew_mean=self.ep_rew_mean[a], episodes=self.ep_count[a]))
        return self

    # ---- state ---------------------------------------------------------------------------------------
    def adam_state(self):
        """(m, v, step): torch views [K, n_params], [K, n_params], [K] of the handle's device memory."""
        m, v, st = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._check(self.lib.qs_ppo_pop_state(self._h, C.byref(m), C.byref(v), C.byref(st)), "qs_ppo_pop_state")
        K, npar = self.params.shape

        class View:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
        with torch.cuda.device(self.device):
            return (torch.as_tensor(View(m.value, (K, npar), "<f4"), device=self.device),
                    torch.as_tensor(View(v.value, (K, npar), "<f4"), device=self.device),
                    torch.as_tensor(View(st.value, (K,), "<i8"), device=self.device))

    def state_dict(self, a: int) -> dict:
        """Agent a's SB3-named policy parameters."""
        return unpack_params(self.params[a].detach().cpu().numpy(), self.obs_dim)

    def save_agent(self, a: int, path: str, template_zip: str | None = None) -> None:
        """Agent a as an SB3 2.6.0 model zip (sb3_compat.save_model_zip): its policy, its Adam state as policy.optimizer.pth, its
        plain hyper-parameters and num_timesteps.  No exact-resume member: QuadPPO.load(path, BatchedQuadEnv(n, ...)) continues
        from it as SB3's PPO.load + learn(reset_num_timesteps=False) does."""
        torch.cuda.synchronize(self.device)
        m, v, step = (t[a].cpu().numpy() for t in self.adam_state())
        opt_sd = sb3_compat.blobs_to_adam_state(m, v, int(step), self.obs_dim, self.hyper["learning_rate"][a])
        data = {"num_timesteps": int(self.num_timesteps), "_n_updates": int(self._n_updates)}
        for k in QuadPPO.HYPER:
            val = self.hyper[k][a] if k in self.hyper else getattr(self, k)
            data[k] = bool(val) if k == "normalize_advantage" else int(val) if k in ("n_steps", "batch_size", "n_epochs") else float(val)
        sb3_compat.save_model_zip(path, self.state_dict(a), opt_sd, data, template_zip)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.qs_ppo_pop_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
