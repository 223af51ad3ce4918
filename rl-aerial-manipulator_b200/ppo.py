"""QuadPPO -- on-device PPO training loop around the batched simulator (SURVEY section 8(f), row 1).

Mirrors `stable_baselines3.PPO("MlpPolicy", env, ...).learn(total_timesteps)` as the reference calls it
(initial-implementation-v1/rl_train_vecN.py:13-36: n_steps=2048, batch_size=128, n_epochs=10, gamma=0.995, gae_lambda=0.9,
clip_range=0.2, ent_coef=0.01, learning_rate=2e-4, net_arch=[128,64,64], Tanh; initial-implementation-v2/rl_train.py:27-56)
with SB3 2.6.0 semantics restated: rollout collection with action clipping and time-limit bootstrapping
(OnPolicyAlgorithm.collect_rollouts), GAE (RolloutBuffer.compute_returns_and_advantage), the clipped surrogate / value /
entropy loss with advantage normalisation, gradient-norm clipping and Adam(eps=1e-5) (PPO.train).

Everything on the hot path is a hand-written kernel behind the C-ABI:
  * rollout: env step (+ fused VecNormalize moments), tcgen05 policy forward, GAE (csrc/qs_gae.cu); time-major buffers [T, N, ...]
    that never leave HBM;
  * update: ONE kernel per minibatch (csrc/qs_ppo.cu, `qs_ppo_update`): gather, forward, loss, backward, global-norm clipping
    and Adam, parameters updated in place in the blob the rollout kernels read.  No torch.nn, no autograd, no torch.optim.
    With the env batch sharded over ranks: `qs_ppo_grad` -> NCCL all-reduce of the 30,7xx gradients -> `qs_ppo_apply`.
torch is the plumbing: device buffers, streams, the epoch permutation, the NCCL collective.
"""
from __future__ import annotations

import ctypes as C
import io
import json
import math

import numpy as np
import torch
import torch.distributed as dist

from . import sb3_compat
from ._cabi import QsPpoHyper, load_library
from .policy import MlpPolicyKernel, H1, H2, H3, NACT, unpack_params


def _bind(lib):
    if getattr(lib, "_gae_bound", False):
        return
    vp = C.c_void_p
    lib.qs_gae.argtypes = [vp, vp, vp, vp, vp, C.c_int, C.c_int64, C.c_float, C.c_float, vp, vp, vp]
    lib.qs_gae.restype = C.c_int
    lib.qs_rollout_record_pre.argtypes = [vp, C.c_int64, C.c_int] + [vp] * 10 + [vp]
    lib.qs_rollout_record_pre.restype = C.c_int
    lib.qs_rollout_record_post.argtypes = [vp, C.c_int64, vp, C.c_int, vp, vp, vp, C.c_float, vp, C.c_double, C.c_float, vp, vp, vp, vp, vp]
    lib.qs_rollout_record_post.restype = C.c_int
    lib.qs_gae_last_error.restype = C.c_char_p
    lib._gae_bound = True


def gae(rewards, values, episode_starts, last_values, last_dones, gamma: float, gae_lambda: float, out=None):
    """advantages, returns = GAE over time-major device buffers [T, N] (qs_gae); out = (advantages, returns) to reuse buffers."""
    lib = load_library()
    _bind(lib)
    T, n = rewards.shape
    adv, ret = out if out is not None else (torch.empty_like(rewards), torch.empty_like(rewards))
    p = lambda t: C.c_void_p(t.data_ptr())
    for t in (rewards, values, episode_starts, last_values, last_dones):
        assert t.is_contiguous() and t.is_cuda
    rc = lib.qs_gae(p(rewards), p(values), p(episode_starts), p(last_values), p(last_dones), T, n, gamma, gae_lambda, p(adv), p(ret),
                    C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"qs_gae failed ({rc}): {lib.qs_gae_last_error().decode()}")
    return adv, ret


def init_state_dict(obs_dim: int, seed: int = 0, log_std_init: float = 0.0) -> dict:
    """SB3 ActorCriticPolicy initialisation: orthogonal weights (gain sqrt(2) trunk, 0.01 action head, 1 value head), zero biases."""
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def ortho(shape, gain):
        # torch.nn.init.orthogonal_: QR of a Gaussian matrix, columns sign-fixed by diag(R)
        rows, cols = shape
        flat = torch.randn((rows, cols), generator=g)
        if rows < cols:
            flat = flat.t()
        q, r = torch.linalg.qr(flat)
        q = q * torch.sign(torch.diagonal(r)).unsqueeze(0)
        if rows < cols:
            q = q.t()
        return (gain * q).contiguous().numpy().astype(np.float32)
    for net in ("policy_net", "value_net"):
        for i, (k_in, k_out) in zip((0, 2, 4), ((obs_dim, H1), (H1, H2), (H2, H3))):
            sd[f"mlp_extractor.{net}.{i}.weight"] = ortho((k_out, k_in), math.sqrt(2))
            sd[f"mlp_extractor.{net}.{i}.bias"] = np.zeros(k_out, np.float32)
    sd["action_net.weight"], sd["action_net.bias"] = ortho((NACT, H3), 0.01), np.zeros(NACT, np.float32)
    sd["value_net.weight"], sd["value_net.bias"] = ortho((1, H3), 1.0), np.zeros(1, np.float32)
    sd["log_std"] = np.full(NACT, log_std_init, np.float32)
    return sd


STAT_KEYS = ("loss", "policy_gradient_loss", "value_loss", "entropy_loss", "grad_norm", "clip_fraction", "approx_kl", "batch_size")


class PpoUpdateKernel:
    """The optimizer: `qs_ppo_*` of include/quadsim.h.  Owns the Adam moments and step count on the device; `params` is the float32
    blob of the rollout kernels (MlpPolicyKernel.params), updated in place."""

    def __init__(self, params: torch.Tensor, obs_dim: int, clip_range=0.2, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5,
                 learning_rate=3e-4, normalize_advantage=True, betas=(0.9, 0.999), eps=1e-5):
        self.lib = load_library()
        self.params, self.obs_dim, self.device = params, int(obs_dim), params.device
        assert params.dtype == torch.float32 and params.is_contiguous() and params.numel() == self.lib.qs_ppo_n_params(self.obs_dim)
        self.hp = QsPpoHyper(clip_range, ent_coef, vf_coef, max_grad_norm, learning_rate, betas[0], betas[1], eps, int(bool(normalize_advantage)), 0)
        h = C.c_void_p()
        self._check(self.lib.qs_ppo_create(self.device.index or 0, self.obs_dim, C.byref(h)), "qs_ppo_create")
        self._h = h
        self.stats = torch.zeros(len(STAT_KEYS), dtype=torch.float32, device=self.device)
        self.grad = torch.zeros_like(params)

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {self.lib.qs_ppo_last_error().decode()}")

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _batch_ptrs(self, obs, act, old_logp, adv, ret, idx):
        for t in (obs, act, old_logp, adv, ret):
            assert t.dtype == torch.float32 and t.is_contiguous() and t.device == self.device
        assert obs.shape[1] == self.obs_dim and act.shape[1] == NACT
        if idx is not None:
            assert idx.dtype == torch.int64 and idx.is_contiguous()
        B = idx.numel() if idx is not None else obs.shape[0]
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        return [p(obs), p(act), p(old_logp), p(adv), p(ret), p(idx), B]

    def update(self, obs, act, old_logp, adv, ret, idx=None):
        """One minibatch update (single rank): gradients, clipping and Adam in one launch."""
        a = self._batch_ptrs(obs, act, old_logp, adv, ret, idx)
        self._check(self.lib.qs_ppo_update(self._h, C.c_void_p(self.params.data_ptr()), *a, C.byref(self.hp),
                                           C.c_void_p(self.stats.data_ptr()), self._stream()), "qs_ppo_update")

    def update_sharded(self, obs, act, old_logp, adv, ret, idx=None, group=None):
        """Data-parallel: local gradient -> average over ranks (NCCL over NVLink) -> clipping + Adam, identical on every rank."""
        a = self._batch_ptrs(obs, act, old_logp, adv, ret, idx)
        self._check(self.lib.qs_ppo_grad(self._h, C.c_void_p(self.params.data_ptr()), *a, C.byref(self.hp), C.c_void_p(self.grad.data_ptr()),
                                         C.c_void_p(self.stats.data_ptr()), self._stream()), "qs_ppo_grad")
        dist.all_reduce(self.grad, group=group)
        self.grad /= dist.get_world_size(group)
        self._check(self.lib.qs_ppo_apply(self._h, C.c_void_p(self.params.data_ptr()), C.c_void_p(self.grad.data_ptr()), C.byref(self.hp),
                                          C.c_void_p(self.stats.data_ptr()), self._stream()), "qs_ppo_apply")

    def gradient(self, obs, act, old_logp, adv, ret, idx=None) -> torch.Tensor:
        """The summed minibatch gradient alone (blob layout), parameters untouched (tests, diagnostics)."""
        a = self._batch_ptrs(obs, act, old_logp, adv, ret, idx)
        self._check(self.lib.qs_ppo_grad(self._h, C.c_void_p(self.params.data_ptr()), *a, C.byref(self.hp), C.c_void_p(self.grad.data_ptr()),
                                         C.c_void_p(self.stats.data_ptr()), self._stream()), "qs_ppo_grad")
        return self.grad

    def adam_state(self):
        """(m, v, step): torch views of the handle's device memory (checkpointing, tests)."""
        m, v, st, g = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._check(self.lib.qs_ppo_state(self._h, C.byref(m), C.byref(v), C.byref(st), C.byref(g)), "qs_ppo_state")
        n = self.params.numel()

        class View:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
        with torch.cuda.device(self.device):
            return (torch.as_tensor(View(m.value, (n,), "<f4"), device=self.device), torch.as_tensor(View(v.value, (n,), "<f4"), device=self.device),
                    torch.as_tensor(View(st.value, (1,), "<i8"), device=self.device))

    def read_stats(self) -> dict:
        return dict(zip(STAT_KEYS, self.stats.tolist()))

    def close(self):
        if self._h:
            self.lib.qs_ppo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class QuadPPO:
    def __init__(self, env, vecnorm=None, state_dict: dict | None = None, n_steps: int = 64, batch_size: int = 65536, n_epochs: int = 10,
                 gamma: float = 0.995, gae_lambda: float = 0.9, clip_range: float = 0.2, ent_coef: float = 0.01, vf_coef: float = 0.5,
                 max_grad_norm: float = 0.5, learning_rate: float = 2e-4, normalize_advantage: bool = True, seed: int = 0,
                 policy_impl: str = "auto", boot_cap: int | None = None, rollout_graph: bool | None = None):
        self.env, self.vecnorm = env, vecnorm
        self.n_steps, self.batch_size, self.n_epochs = n_steps, batch_size, n_epochs
        self.gamma, self.gae_lambda = gamma, gae_lambda
        self.clip_range, self.ent_coef, self.vf_coef, self.max_grad_norm = clip_range, ent_coef, vf_coef, max_grad_norm
        self.learning_rate, self.normalize_advantage = learning_rate, normalize_advantage
        dev, n, d = env.device, env.n_envs, env.obs_dim
        sd = state_dict or init_state_dict(d, seed)
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.policy = MlpPolicyKernel(sd, d, dev, impl=policy_impl)
        # second set of output buffers for the time-limit bootstrap / last-value forwards (other batch sizes): same parameter blob
        self._aux = MlpPolicyKernel(sd, d, dev, impl=policy_impl)
        self._aux.params = self.policy.params
        self.opt = PpoUpdateKernel(self.policy.params, d, clip_range=clip_range, ent_coef=ent_coef, vf_coef=vf_coef, max_grad_norm=max_grad_norm,
                                   learning_rate=learning_rate, normalize_advantage=normalize_advantage)
        self.gen = torch.Generator(device=dev).manual_seed(seed + 1000 * (dist.get_rank() if dist.is_initialized() else 0))
        T = n_steps
        f32 = dict(dtype=torch.float32, device=dev)
        self.obs = torch.empty((T, n, d), **f32)
        self.actions = torch.empty((T, n, NACT), **f32)
        self.values, self.logp, self.rewards = torch.empty((T, n), **f32), torch.empty((T, n), **f32), torch.empty((T, n), **f32)
        self.advantages, self.returns = torch.empty((T, n), **f32), torch.empty((T, n), **f32)
        self.episode_starts = torch.zeros((T, n), dtype=torch.uint8, device=dev)
        self._noise = torch.empty((n, NACT), **f32)
        # slots for time-limit bootstraps per step: every env up to 65,536 envs (no overflow possible), a sixteenth of the shard above
        # that (more than 6 % of a shard hitting the limit in the same step raises after the rollout; `boot_cap` overrides)
        self._boot_cap = int(boot_cap) if boot_cap else (n if n <= 65536 else max(65536, n // 16))
        self._boot_slots = torch.arange(self._boot_cap, device=dev)
        self._boot_zero = torch.zeros((), **f32)
        self._boot_overflow = torch.zeros((), dtype=torch.bool, device=dev)
        self._last_dones = torch.ones(n, dtype=torch.uint8, device=dev)
        self._last_obs = None
        # rollout_graph: one collection step (about thirty small launches of bookkeeping around the two kernels) captured ONCE as a
        # CUDA graph and replayed per step -- at the reference's 8 envs x 2048 steps a collection is bound by the host's launch path
        # (profiles/r02/ppo_ref_hparams_breakdown.txt), not by the device.  None: on for a single rank.
        self._use_graph = (self.world == 1) if rollout_graph is None else bool(rollout_graph)
        self._graph = None
        self._t = torch.zeros(1, dtype=torch.int64, device=dev)             # the step's slot in the rollout buffers (device: graph replays)
        self._st_obs = torch.empty((n, d), **f32)
        self._st_rew = torch.empty(n, **f32)
        self._rec_ws = torch.zeros(2 * 1024 + 1, dtype=torch.float64, device=dev)   # qs_rollout_record_post workspace (QS_RECORD_MAX_BLOCKS)
        self.num_timesteps = 0
        self._n_updates = 0
        self._ep_stats = torch.zeros(2, dtype=torch.float64, device=dev)
        self._zero = torch.zeros((), dtype=torch.float64, device=dev)
        self.ep_rew_mean, self.ep_count = float("nan"), 0

    # ---- rollout -------------------------------------------------------------------------------------
    def _forward(self, obs_raw, noise, obs_norm_out=None, policy=None):
        stats = self.vecnorm.obs_rms.stats if (self.vecnorm is not None and self.vecnorm.norm_obs) else None
        eps, clip = (self.vecnorm.epsilon, self.vecnorm.clip_obs) if self.vecnorm is not None else (1e-8, 10.0)
        return (policy or self.policy).forward(obs_raw, noise, norm_stats=stats, norm_eps=eps, norm_clip=clip, obs_norm_out=obs_norm_out)

    def _bootstrap_truncated(self, out, rew):
        """TimeLimit.truncated: rew += gamma * V(terminal_obs) for the envs that hit the time limit only -- without a host round trip.
        Up to 65,536 envs the critic simply runs on every env's terminal_obs row and the result is masked (rows of envs that did not
        finish hold an older episode's terminal observation: finite, and discarded by the where); above, the truncated envs are
        compacted into a FIXED number of slots (nonzero_static; unused slots point at env 0 and add zero), so nothing waits for a count."""
        trunc_only = (out.flags & 3) == 2
        if self._boot_cap >= self.env.n_envs:
            tv = self._forward(out.terminal_obs, None, policy=self._aux)[1]
            rew.add_(torch.where(trunc_only, self.gamma * tv, self._boot_zero))
            return
        cnt = trunc_only.sum()
        idx = torch.nonzero_static(trunc_only, size=self._boot_cap, fill_value=0)[:, 0]
        tv = self._forward(out.terminal_obs.index_select(0, idx), None, policy=self._aux)[1]
        rew.index_add_(0, idx, torch.where(self._boot_slots < cnt, self.gamma * tv, self._boot_zero))
        self._boot_overflow |= cnt > self._boot_cap

    def _graph_step(self):
        """One collection step with every address fixed (what _collect_eager does per step, with the slot of the rollout buffers taken
        from the device-resident counter self._t through index_copy_): capturable, and the body of the replayed graph."""
        env, vn = self.env, self.vecnorm
        self._noise.normal_(generator=self.gen)
        raw = env.obs
        use_norm = vn is not None and vn.norm_obs
        a, v, lp = self._forward(raw, self._noise, self._st_obs if use_norm else None)
        if self._boot_cap >= env.n_envs:
            return self._graph_step_kernels(raw, use_norm, a, v, lp)
        t = self._t
        self.obs.index_copy_(0, t, (self._st_obs if use_norm else raw).unsqueeze(0))
        self.actions.index_copy_(0, t, a.unsqueeze(0))
        self.values.index_copy_(0, t, v.unsqueeze(0))
        self.logp.index_copy_(0, t, lp.unsqueeze(0))
        self.episode_starts.index_copy_(0, t, self._last_dones.unsqueeze(0))
        out = env.step(self.policy.actions_clipped)
        if vn is not None and vn.training:
            if vn.norm_obs:
                vn.obs_rms.update_from_moments()
            vn.update_returns(out)
        if vn is not None and vn.norm_reward:
            torch.clamp(out.reward / torch.sqrt(vn.ret_rms.var[0] + vn.epsilon), -vn.clip_reward, vn.clip_reward, out=self._st_rew)
        else:
            self._st_rew.copy_(out.reward)
        self._bootstrap_truncated(out, self._st_rew)
        self.rewards.index_copy_(0, t, self._st_rew.unsqueeze(0))
        done = (out.flags & 3) != 0
        self._last_dones.copy_(done)
        self._ep_stats[0] += torch.where(done, out.ep_return.double(), self._zero).sum()
        self._ep_stats[1] += done.sum()
        self._t.add_(1)

    def _graph_step_kernels(self, raw, use_norm, a, v, lp):
        """The rest of _graph_step with the bookkeeping in two kernels (qs_rollout_record_pre / _post: RolloutBuffer.add, reward
        normalisation, time-limit bootstrap, last dones, episode statistics, slot counter) instead of ~25 small torch launches; the
        critic runs on every env's terminal_obs row (shards up to 65,536 envs).  Same float32 arithmetic as the torch expressions."""
        env, vn = self.env, self.vecnorm
        lib = load_library()
        _bind(lib)
        p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None
        st = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
        n = env.n_envs
        rc = lib.qs_rollout_record_pre(p(self._t), n, env.obs_dim, p(self._st_obs if use_norm else raw), p(a), p(v), p(lp), p(self._last_dones),
                                       p(self.obs), p(self.actions), p(self.values), p(self.logp), p(self.episode_starts), st)
        if rc != 0:
            raise RuntimeError(f"qs_rollout_record_pre failed ({rc}): {lib.qs_gae_last_error().decode()}")
        out = env.step(self.policy.actions_clipped)
        if vn is not None and vn.training:
            if vn.norm_obs:
                vn.obs_rms.update_from_moments()
            vn.update_returns(out)
        tv = self._forward(out.terminal_obs, None, policy=self._aux)[1]
        norm_r = vn is not None and vn.norm_reward
        rc = lib.qs_rollout_record_post(p(self._t), n, p(out.reward), int(out.reward.dtype == torch.float64), p(out.flags), p(out.ep_return), p(tv),
                                        float(self.gamma), C.c_void_p(vn.ret_rms.stats.data_ptr() + 16) if norm_r else None,
                                        float(vn.epsilon) if norm_r else 0.0, float(vn.clip_reward) if norm_r else 0.0, p(self.rewards),
                                        p(self._last_dones), p(self._ep_stats), p(self._rec_ws), st)
        if rc != 0:
            raise RuntimeError(f"qs_rollout_record_post failed ({rc}): {lib.qs_gae_last_error().decode()}")

    def _collect_graph(self) -> bool:
        """The n_steps of a collection as replays of one captured step.  The first two steps of the first collection run eagerly
        (lazy initialisation must not happen under capture); they are real steps.  False: not applicable, collect eagerly."""
        env = self.env
        if self.n_steps < 4 or self._last_obs.data_ptr() != env.obs.data_ptr():
            return False
        vn = self.vecnorm
        key = (vn is not None, bool(vn and vn.training), bool(vn and vn.norm_obs), bool(vn and vn.norm_reward), float(self.gamma), self.n_steps)
        if self._graph is not None and self._graph[1] != key:
            self._graph = None                                   # a setting the captured step depends on has changed
        self._t.zero_()
        done = 0
        if self._graph is None:
            for _ in range(2):
                self._graph_step()
            done = 2
            torch.cuda.synchronize(env.device)
            try:
                g = torch.cuda.CUDAGraph()
                g.register_generator_state(self.gen)
                with torch.cuda.graph(g):
                    self._graph_step()
            except Exception as exc:  # noqa: BLE001 -- a launch-mode optimisation only: the same step body goes on eagerly
                import warnings
                warnings.warn(f"QuadPPO: the collection step could not be captured as a CUDA graph ({exc}); collecting eagerly")
                torch.cuda.synchronize(env.device)
                self._use_graph = False
                for _ in range(done, self.n_steps):
                    self._graph_step()
                self._last_obs = env.obs
                return True
            self._graph = (g, key)
        g = self._graph[0]
        for _ in range(done, self.n_steps):
            g.replay()
        self._last_obs = env.obs
        return True

    def collect_rollouts(self):
        env, vn = self.env, self.vecnorm
        if self._last_obs is None:
            self._last_obs = env.reset()
            if vn is not None and vn.norm_obs and vn.training:
                vn.obs_rms.update(self._last_obs)                # VecNormalize.reset() updates the statistics too
                self._attach_moments()
        self._ep_stats.zero_()
        if not (self._use_graph and self._collect_graph()):
            self._collect_eager()
        self._finish_rollout()

    def _attach_moments(self):
        """From here on the step kernel reduces its own observations and, where one launch can do it (one GPU, or several over the
        peer-memory exchange), the kernel that finishes them also merges them into the running statistics."""
        rms = self.vecnorm.obs_rms
        rms.attach(self.env, merge=(rms._gathered is None or rms.exchange == "peer"))

    def _collect_eager(self):
        env, vn = self.env, self.vecnorm
        for t in range(self.n_steps):
            self._noise.normal_(generator=self.gen)
            raw = self._last_obs
            norm_out = self.obs[t] if vn is not None and vn.norm_obs else None
            a, v, lp = self._forward(raw, self._noise, norm_out)
            if norm_out is None:
                self.obs[t].copy_(raw)
            self.actions[t].copy_(a)
            self.values[t].copy_(v)
            self.logp[t].copy_(lp)
            self.episode_starts[t].copy_(self._last_dones)
            out = env.step(self.policy.actions_clipped)            # SB3 clips to the action box before env.step, stores the unclipped
            if vn is not None and vn.training:
                if vn.norm_obs:
                    vn.obs_rms.update_from_moments()
                vn.update_returns(out)
            if vn is not None and vn.norm_reward:                   # VecNormalize.normalize_reward, after this step's ret_rms update
                torch.clamp(out.reward / torch.sqrt(vn.ret_rms.var[0] + vn.epsilon), -vn.clip_reward, vn.clip_reward, out=self.rewards[t])
            else:
                self.rewards[t].copy_(out.reward)
            self._bootstrap_truncated(out, self.rewards[t])
            done = (out.flags & 3) != 0
            self._last_dones.copy_(done)                            # in place: the captured step (rollout_graph) reads this buffer
            self._ep_stats[0] += torch.where(done, out.ep_return.double(), self._zero).sum()     # Monitor-style episode returns,
            self._ep_stats[1] += done.sum()                                                     # reduced on device
            self._last_obs = out.obs

    def _finish_rollout(self):
        env, vn = self.env, self.vecnorm
        last_values = self._forward(self._last_obs, None, policy=self._aux)[1]
        gae(self.rewards, self.values, self.episode_starts, last_values, self._last_dones, self.gamma, self.gae_lambda,
            out=(self.advantages, self.returns))
        if vn is not None and vn.norm_obs and vn.obs_rms.exchange_failed():
            raise RuntimeError("VecNormalize moment exchange timed out waiting for a rank: the running statistics are incomplete")
        if bool(self._boot_overflow):
            raise RuntimeError(f"more than {self._boot_cap} envs hit the time limit in one step: raise QuadPPO._boot_cap")
        self.num_timesteps += self.n_steps * env.n_envs * self.world
        s, c = self._ep_stats.tolist()
        self.ep_rew_mean = s / c if c > 0 else float("nan")     # mean return of the episodes that finished in this rollout
        self.ep_count = int(c)

    # ---- update --------------------------------------------------------------------------------------
    def train(self) -> dict:
        """PPO.train: n_epochs passes over the rollout buffer in shuffled minibatches, the ragged last one included (as SB3's
        RolloutBuffer.get does).  One kernel launch per minibatch; the only host sync is the statistics read at the end."""
        T, n = self.rewards.shape
        total = T * n
        flat = lambda x: x.reshape(total, *x.shape[2:])
        obs, act, oldlp, adv, ret = map(flat, (self.obs, self.actions, self.logp, self.advantages, self.returns))
        bs = min(self.batch_size, total)
        for epoch in range(self.n_epochs):
            perm = torch.randperm(total, device=obs.device, generator=self.gen)
            for start in range(0, total, bs):
                idx = perm[start:start + bs]
                if self.world > 1:
                    self.opt.update_sharded(obs, act, oldlp, adv, ret, idx)
                else:
                    self.opt.update(obs, act, oldlp, adv, ret, idx)
        self._n_updates += self.n_epochs
        return {k: v for k, v in self.opt.read_stats().items()}

    def learn(self, total_timesteps: int, log=None, callback=None):
        """Train until num_timesteps reaches total_timesteps (SB3's learn with reset_num_timesteps=False).  callback: an
        evaluation.EvalCallback or CheckpointCallback, a list of them (called in order after every train(); their results join
        the log dict), or None."""
        callbacks = [] if callback is None else list(callback) if isinstance(callback, (list, tuple)) else [callback]
        for cb in callbacks:
            cb.init_callback(self)
        while self.num_timesteps < total_timesteps:
            self.collect_rollouts()
            info = self.train()
            for cb in callbacks:
                info.update(cb.after_train(self))
            if log:
                log(dict(info, timesteps=self.num_timesteps, ep_rew_mean=self.ep_rew_mean, episodes=self.ep_count))
        return self

    def state_dict(self) -> dict:
        """SB3-named policy parameters (feed to sb3_compat.save_policy_zip)."""
        return unpack_params(self.policy.params.detach().cpu().numpy(), self.env.obs_dim)

    # ---- checkpoints ---------------------------------------------------------------------------------
    HYPER = ("n_steps", "batch_size", "n_epochs", "gamma", "gae_lambda", "clip_range", "ent_coef", "vf_coef", "max_grad_norm",
             "learning_rate", "normalize_advantage")

    def _resume_config(self) -> dict:
        """What the exact-resume state depends on besides the hyper-parameters: the env's configuration and the VecNormalize mode."""
        env, c, vn = self.env, self.env.cfg, self.vecnorm
        return {"env_version": env.env_version, "precision": env.precision, "integrator": env.integrator, "substeps": int(c.substeps),
                "obs_scaled": bool(c.obs_scaled), "action_scale_f32": bool(c.action_scale_f32), "auto_reset": bool(c.auto_reset),
                "n_envs": env.n_envs, "env_id_offset": int(c.env_id_offset), "seed": env.seed,
                "v2_random_waypoints": bool(c.v2_random_waypoints),
                "dynamics_randomization": json.loads(json.dumps(env.dynamics_randomization, sort_keys=True)),
                "vecnorm": None if vn is None else {"norm_obs": bool(vn.norm_obs), "norm_reward": bool(vn.norm_reward), "training": bool(vn.training)}}

    def _resume_bytes(self) -> bytes:
        """Every piece of device and host state that crosses an iteration boundary, as an .npz (see DESIGN "Checkpoints and resume")."""
        env, vn = self.env, self.vecnorm
        host = lambda t: t.detach().cpu().numpy()
        m, v, step = self.opt.adam_state()
        a = {"config": np.array(json.dumps(self._resume_config(), sort_keys=True)), "params": host(self.policy.params), "adam_m": host(m),
             "adam_v": host(v), "adam_step": host(step), "generator": self.gen.get_state().numpy(),
             "progress": np.array([self.num_timesteps, self.ep_count, self._n_updates], np.int64), "ep_rew_mean": np.float64(self.ep_rew_mean)}
        if self._last_obs is not None:                       # collection has started: the env is mid-episode
            a.update({f"env.{k}": host(t) for k, t in env.get_state().items()})
            a["env_obs"], a["last_dones"] = host(env.obs), host(self._last_dones)
            if env.dynamics_randomization is not None:
                a["dynamics"] = host(env._dyn_rows())
        if vn is not None:
            a["obs_rms"], a["ret_rms"], a["returns"] = host(vn.obs_rms.stats), host(vn.ret_rms.stats), host(vn.returns)
            if self._last_obs is not None and vn.norm_obs and vn.training:
                a["obs_moments"] = host(vn.obs_rms._moments)
        buf = io.BytesIO()
        np.savez(buf, **a)
        return buf.getvalue()

    def _restore(self, a) -> None:
        """Inverse of _resume_bytes on a freshly built QuadPPO: no env.reset(), no statistics update."""
        want, have = json.loads(str(a["config"])), self._resume_config()
        for k in want:
            if want[k] != have.get(k):
                raise ValueError(f"checkpoint was saved with {k} = {want[k]!r}, this env has {have.get(k)!r} "
                                 "(resume_env_state=False resumes with a fresh env reset instead)")
        env, vn = self.env, self.vecnorm
        dev = lambda x: torch.from_numpy(np.asarray(x)).to(env.device)
        m, v, step = self.opt.adam_state()
        self.policy.params.copy_(dev(a["params"]))
        m.copy_(dev(a["adam_m"]))
        v.copy_(dev(a["adam_v"]))
        step.copy_(dev(a["adam_step"]))
        self.gen.set_state(torch.from_numpy(a["generator"]))
        self.num_timesteps, self.ep_count, self._n_updates = (int(x) for x in a["progress"])
        self.ep_rew_mean = float(a["ep_rew_mean"])
        if vn is not None:
            vn.obs_rms.stats.copy_(dev(a["obs_rms"]))
            vn.ret_rms.stats.copy_(dev(a["ret_rms"]))
            vn.returns.copy_(dev(a["returns"]))
        if "env_obs" not in a:
            return                                           # saved before the first collection: it resets the env as usual
        env.set_state(**{k[4:]: a[k] for k in a.files if k.startswith("env.")})
        if "dynamics" in a:                                  # after the pool: arming drew parameters for the episodes it found
            d = a["dynamics"]
            env.set_dynamics(mass_scale=d[:, 0], inertia_scale=d[:, 1], thrust_scale=d[:, 2:6], wind=d[:, 6:9])
        env.obs.copy_(dev(a["env_obs"]))
        self._last_dones.copy_(dev(a["last_dones"]))
        self._last_obs = env.obs
        if "obs_moments" in a:
            self._attach_moments()                           # as collect_rollouts does after its first reset ...
            vn.obs_rms._moments.copy_(dev(a["obs_moments"]))  # ... but centred where the interrupted run's next step would centre
        torch.cuda.synchronize(env.device)

    def save(self, path: str, template_zip: str | None = None, vecnormalize_path: str | None = None) -> None:
        """model.save(path): an SB3 2.6.0 model zip (sb3_compat.save_model_zip) with the policy, the Adam state as
        policy.optimizer.pth and the plain hyper-parameters in `data`, plus the exact-resume member (sb3_compat.RESUME_MEMBER)
        that QuadPPO.load uses to continue bit for bit.  template_zip: an SB3 zip whose pickled `data` entries are kept (see
        save_model_zip).  vecnormalize_path: also write the VecNormalize statistics as an SB3 vec_normalize.pkl.  Single rank."""
        if self.world > 1:
            raise ValueError("QuadPPO.save is single-rank only")
        if vecnormalize_path is not None and self.vecnorm is None:
            raise ValueError("vecnormalize_path given, but this QuadPPO has no VecNormalize")
        torch.cuda.synchronize(self.env.device)
        d = self.env.obs_dim
        m, v, step = (t.cpu().numpy() for t in self.opt.adam_state())
        opt_sd = sb3_compat.blobs_to_adam_state(m, v, int(step[0]), d, self.learning_rate)
        data = {"num_timesteps": int(self.num_timesteps), "_n_updates": int(self._n_updates)}
        for k in self.HYPER:
            val = getattr(self, k)
            data[k] = bool(val) if k == "normalize_advantage" else int(val) if k in ("n_steps", "batch_size", "n_epochs") else float(val)
        sb3_compat.save_model_zip(path, self.state_dict(), opt_sd, data, template_zip, extra={sb3_compat.RESUME_MEMBER: self._resume_bytes()})
        if vecnormalize_path is not None:
            vn = self.vecnorm
            sb3_compat.save_vecnormalize_pkl(vecnormalize_path, dict(vn.state_dict(), training=vn.training), self.env.n_envs, d)

    @classmethod
    def load(cls, path: str, env, vecnorm=None, resume_env_state: bool = True, **overrides) -> "QuadPPO":
        """PPO.load(path, env): a QuadPPO on `env` with the zip's parameters, Adam state and num_timesteps; hyper-parameters from
        the zip's `data` (plain entries; e.g. the reference's batch_size=128 is kept unless overridden), `overrides` (any QuadPPO
        keyword) win.  When the zip carries QuadPPO.save's resume member and resume_env_state is True, training continues exactly
        where it was saved (env, VecNormalize statistics, generator): an env whose configuration differs raises ValueError.
        Otherwise (an SB3 zip, or resume_env_state=False) it resumes as PPO.load + learn(reset_num_timesteps=False) does: the env
        is reset at the first collection, and VecNormalize statistics are the caller's (load_vecnormalize_pkl +
        DeviceVecNormalize.load_state_dict).  Single rank."""
        if dist.is_initialized() and dist.get_world_size() > 1:
            raise ValueError("QuadPPO.load is single-rank only")
        z = sb3_compat.read_model_zip(path)
        data, policy_sd = z["data"], z["policy"]
        kw = {k: data[k] for k in cls.HYPER if k in data and not isinstance(data[k], dict)}
        kw.update(overrides)
        ppo = cls(env, vecnorm, state_dict=policy_sd, **kw)
        if z["optimizer"] is not None:
            m, v, step, group = sb3_compat.adam_state_to_blobs(z["optimizer"], list(policy_sd), env.obs_dim)
            if tuple(group.get("betas", (0.9, 0.999))) != (0.9, 0.999) or float(group.get("eps", 1e-5)) != 1e-5:
                raise ValueError(f"optimizer has betas {group.get('betas')} and eps {group.get('eps')}; the update kernel runs "
                                 "SB3's Adam(betas=(0.9, 0.999), eps=1e-5)")
            dm, dv, dstep = ppo.opt.adam_state()
            dm.copy_(torch.from_numpy(m))
            dv.copy_(torch.from_numpy(v))
            dstep.fill_(step)
        ppo.num_timesteps = int(data.get("num_timesteps", 0))
        ppo._n_updates = int(data.get("_n_updates", 0))
        if resume_env_state and sb3_compat.RESUME_MEMBER in z["members"]:
            with np.load(io.BytesIO(z["members"][sb3_compat.RESUME_MEMBER]), allow_pickle=False) as a:
                ppo._restore(a)
        torch.cuda.synchronize(env.device)
        return ppo
