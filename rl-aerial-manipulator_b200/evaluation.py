"""evaluate_policy and EvalCallback on the device.

Replaces stable_baselines3.common.evaluation.evaluate_policy (SB3 2.6.0; reference call site
initial-implementation-v1/rl_train_vecN.py:42, `evaluate_policy(model, env, 10)`) and SB3's EvalCallback and CheckpointCallback
for QuadPPO.

Every evaluation step is three launches: the shipped policy forward (`MlpPolicyKernel.forward`, or `forward_sampled` with in-kernel
Philox noise), the shipped env step (`BatchedQuadEnv.step` on the box-clipped actions, as SB3's `predict` clips) and
`qs_eval_record` (csrc/qs_eval.cu), which applies SB3's episode selection on the device.  `poll_every` steps are captured once as a
CUDA graph and replayed; after each replay the host reads one word (`remaining`) and stops at zero.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import warnings
from dataclasses import dataclass

import numpy as np
import torch

from . import _cabi
from ._cabi import load_library
from .policy import IMPL, MlpPolicyKernel, unpack_params

MAX_STEPS = {1: 1200, 2: 2000}       # the envs' time limits (csrc/qs_env.cuh EnvTraits): no episode is longer than MAX_STEPS + 1


def targets(n_eval_episodes: int, n_global: int, env_ids) -> np.ndarray:
    """SB3's per-env target (n_eval_episodes + i) // n_envs, in the closed form of csrc/qs_eval.cuh."""
    q, r = divmod(int(n_eval_episodes), int(n_global))
    return q + (np.asarray(env_ids, dtype=np.int64) >= n_global - r)


def first_slot(n_eval_episodes: int, n_global: int, env_ids) -> np.ndarray:
    """base(i): the slot of env i's first recorded episode among all n_eval_episodes (sum of the targets of the envs before it)."""
    q, r = divmod(int(n_eval_episodes), int(n_global))
    i = np.asarray(env_ids, dtype=np.int64)
    return q * i + np.maximum(0, i - (n_global - r))


@dataclass
class EvalResult:
    """The recorded episodes as device tensors, in SB3's order (completion step, then global env id):
    ep_return f64 (Monitor 'r', not rounded), ep_length i32 (Monitor 'l'), flags u8 (QS_FLAG_* of the finishing step),
    step i32 (the 0-based evaluation step in which the episode finished), env_id i64 (global)."""
    ep_return: torch.Tensor
    ep_length: torch.Tensor
    flags: torch.Tensor
    step: torch.Tensor
    env_id: torch.Tensor
    n_global: int
    steps: int = 0           # env steps this evaluation ran (several ranks: the most any rank ran)

    def __post_init__(self):
        order = torch.argsort(self.step.to(torch.int64) * self.n_global + self.env_id)
        for f in ("ep_return", "ep_length", "flags", "step", "env_id"):
            setattr(self, f, getattr(self, f)[order])

    @staticmethod
    def concat(results: list["EvalResult"]) -> "EvalResult":
        """Merge the results of the shards of one evaluation (each rank's evaluate(..., n_global=G)); the tensors are moved to the
        first result's device.  Gathering them across processes is the caller's."""
        dev = results[0].ep_return.device
        cat = lambda f: torch.cat([getattr(r, f).to(dev) for r in results])
        return EvalResult(cat("ep_return"), cat("ep_length"), cat("flags"), cat("step"), cat("env_id"), results[0].n_global,
                          max(r.steps for r in results))

    def episode_rewards(self) -> list[float]:
        """Monitor's info['episode']['r'] values: rounded to 6 decimals, SB3's order."""
        return [round(float(r), 6) for r in self.ep_return.cpu().numpy()]

    def episode_lengths(self) -> list[int]:
        return [int(x) for x in self.ep_length.cpu().numpy()]

    def _rate(self, mask: torch.Tensor) -> float:
        return float(mask.double().mean()) if mask.numel() else float("nan")

    @property
    def success_rate(self) -> float:
        """info['success'] on a terminated episode (QS_FLAG_SUCCESS & QS_FLAG_TERMINATED)."""
        return self._rate(self._success())

    def _success(self) -> torch.Tensor:
        both = _cabi.FLAG_SUCCESS | _cabi.FLAG_TERMINATED
        return (self.flags & both) == both

    @property
    def crash_rate(self) -> float:
        return self._rate((self.flags & _cabi.FLAG_CRASHED) != 0)

    @property
    def oob_rate(self) -> float:
        return self._rate((self.flags & _cabi.FLAG_OOB) != 0)

    @property
    def truncation_rate(self) -> float:
        return self._rate((self.flags & _cabi.FLAG_TRUNCATED) != 0)

    @property
    def mean_length_successful(self) -> float:
        s = self._success()
        return float(self.ep_length[s].double().mean()) if bool(s.any()) else float("nan")


def evaluate(policy: MlpPolicyKernel, env, n_eval_episodes: int = 10, deterministic: bool = True, vecnorm=None, noise_seed: int = 0,
             n_global: int | None = None, poll_every: int = 64, warn: bool = True) -> EvalResult:
    """evaluate_policy's episodes as an EvalResult (see evaluate_policy for the arguments)."""
    lib = load_library()
    n, off = env.n_envs, int(env.cfg.env_id_offset)
    G = n if n_global is None else int(n_global)
    E = int(n_eval_episodes)
    if E < 1:
        raise ValueError("n_eval_episodes must be >= 1")
    if not 0 <= off <= G - n:
        raise ValueError(f"env ids [{off}, {off + n}) do not fit in n_global = {G}")
    if int(poll_every) < 1:
        raise ValueError("poll_every must be >= 1")
    if policy.obs_dim != env.obs_dim or policy.device != env.device:
        raise ValueError("policy and env differ in observation size or device")
    tgt_max = int(targets(E, G, [off + n - 1])[0])        # targets do not decrease with the env id
    if tgt_max > 1 and not bool(env.cfg.auto_reset):
        raise ValueError(f"n_eval_episodes = {E} over {G} envs needs {tgt_max} episodes from some env, but the env does not auto-reset "
                         "(auto_reset=False: evaluate one episode per env, n_eval_episodes <= n_envs)")
    stats, eps, clip = None, 1e-8, 10.0
    if vecnorm is not None and vecnorm.norm_obs:
        stats, eps, clip = vecnorm.obs_rms.stats, float(vecnorm.epsilon), float(vecnorm.clip_obs)
    dev = env.device
    first, last = first_slot(E, G, [off, off + n])
    slots = int(last - first)
    m = max(slots, 1)
    count = torch.zeros(n, dtype=torch.int32, device=dev)
    state = torch.zeros(_cabi.EVAL_STATE_WORDS, dtype=torch.int32, device=dev)
    ret = torch.zeros(m, dtype=torch.float64, device=dev)
    length = torch.zeros(m, dtype=torch.int32, device=dev)
    flags = torch.zeros(m, dtype=torch.uint8, device=dev)
    step = torch.zeros(m, dtype=torch.int32, device=dev)
    a = _cabi.QsEvalArgs()
    a.n, a.env_id_offset, a.n_global, a.n_eval_episodes = n, off, G, E
    a.return_is_f64 = int(env.ep_return.dtype == torch.float64)
    p = lambda t: t.data_ptr()
    a.flags, a.ep_return, a.ep_len = p(env.flags), p(env.ep_return), p(env.ep_len)
    a.count, a.state, a.ret_out, a.len_out, a.flags_out, a.step_out = p(count), p(state), p(ret), p(length), p(flags), p(step)
    stream = lambda: C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def check(rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {lib.qs_eval_last_error().decode()}")

    if not deterministic:
        if getattr(policy, "_philox_counter", None) is None:
            policy._philox_counter = torch.zeros(2, dtype=torch.int64, device=dev)
        policy._philox_counter.zero_()              # noise = f(noise_seed, global env id, evaluation step): the same seed reproduces

    def one_step():
        if deterministic:
            policy.forward(env.obs, None, norm_stats=stats, norm_eps=eps, norm_clip=clip)
        else:
            policy.forward_sampled(env.obs, noise_seed, off, norm_stats=stats, norm_eps=eps, norm_clip=clip)
        env.step(policy.actions_clipped)
        check(lib.qs_eval_record(C.byref(a), stream()), "qs_eval_record")

    env.reset()
    check(lib.qs_eval_begin(C.byref(a), stream()), "qs_eval_begin")
    P = int(poll_every)
    bound = math.ceil(tgt_max * (MAX_STEPS[env.env_version] + 1) / P) * P
    remaining = torch.empty(1, dtype=torch.int32).pin_memory()
    ev = torch.cuda.Event()

    def poll() -> int:
        remaining.copy_(state[1:2], non_blocking=True)
        ev.record(torch.cuda.current_stream(dev))
        ev.synchronize()
        return int(remaining[0])

    steps = 2                                       # eager first steps: lazy allocations never happen under capture
    for _ in range(steps):
        one_step()
    graph = None
    if poll() != 0:
        torch.cuda.synchronize(dev)
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for _ in range(P):
                    one_step()
        except Exception as exc:  # noqa: BLE001 -- a launch-mode optimisation only: the same steps run eagerly
            if warn:
                warnings.warn(f"evaluate_policy: the evaluation steps could not be captured as a CUDA graph ({exc}); stepping eagerly")
            torch.cuda.synchronize(dev)
            graph = None
        while True:
            if steps >= bound:
                raise RuntimeError(f"evaluation did not finish within {bound} steps (the time limit bounds every episode): "
                                   f"{int(state[1])} envs still below their target")
            if graph is not None:
                graph.replay()
            else:
                for _ in range(P):
                    one_step()
            steps += P
            if poll() == 0:
                break
    env_id = torch.from_numpy(np.repeat(np.arange(off, off + n), targets(E, G, np.arange(off, off + n)))).to(dev)
    return EvalResult(ret[:slots], length[:slots], flags[:slots], step[:slots], env_id, G, steps)


def evaluate_policy(policy: MlpPolicyKernel, env, n_eval_episodes: int = 10, deterministic: bool = True,
                    return_episode_rewards: bool = False, reward_threshold: float | None = None, vecnorm=None, noise_seed: int = 0,
                    n_global: int | None = None, poll_every: int = 64, warn: bool = True, full: bool = False, *,
                    render: bool = False, callback=None):
    """stable_baselines3.common.evaluation.evaluate_policy for a MlpPolicyKernel on a BatchedQuadEnv, on the device.

    Starts with env.reset(); env i records its first (n_eval_episodes + i) // n_global finished episodes (Monitor's return and
    length), and the loop runs until every env has.  deterministic: the mean action (`forward`), else Gaussian noise drawn in the
    kernel from (noise_seed, global env id, step) -- the same seed gives the same evaluation.  Actions are clipped to the action box.
    vecnorm: a DeviceVecNormalize whose observation statistics are applied, read-only; the returns are the env's raw Monitor
    returns, as SB3's are under VecNormalize.  A dynamics-randomised env flies each episode with the airframe drawn for it.
    n_global: envs over all ranks when `env` is one shard (env_id_offset set): this rank records exactly the episodes the
    unsharded batch would give its envs; merge the ranks' EvalResults with EvalResult.concat.
    poll_every: steps per CUDA-graph replay between reads of the one host word that says whether the evaluation is done.
    warn: warn when the steps cannot be captured as a CUDA graph and run eagerly.

    Returns (mean, std) of the episode returns, or (returns, lengths) in SB3's order with return_episode_rewards (returns rounded to 6
    decimals, as Monitor does), or the EvalResult with full=True.  reward_threshold: `assert mean > reward_threshold`, as SB3 does.
    render and callback (SB3's per-step hooks) are not supported: the steps run on the device without visiting the host."""
    if render or callback is not None:
        raise ValueError("evaluate_policy: render and callback are not supported (the evaluation steps never visit the host)")
    res = evaluate(policy, env, n_eval_episodes, deterministic, vecnorm, noise_seed, n_global, poll_every, warn)
    if full:
        return res
    rewards, lengths = res.episode_rewards(), res.episode_lengths()
    mean_reward, std_reward = float(np.mean(rewards)), float(np.std(rewards))
    if reward_threshold is not None:
        assert mean_reward > reward_threshold, f"Mean reward below threshold: {mean_reward:.2f} < {reward_threshold:.2f}"
    if return_episode_rewards:
        return rewards, lengths
    return mean_reward, std_reward


def _vec_steps(ppo) -> int:
    return ppo.num_timesteps // (ppo.env.n_envs * ppo.world)


def _crossed(ppo, freq: int, bucket: int):
    """(due, new bucket): due after the first train() that crosses a multiple of `freq` vec-env steps.  SB3's callbacks fire
    mid-rollout; here the collection is one replayed CUDA graph and is not split, so they fire after the train() that follows."""
    b = _vec_steps(ppo) // freq
    return b != bucket, b


class EvalCallback:
    """stable_baselines3 EvalCallback for QuadPPO.learn(callback=...): evaluates the current policy on `eval_env` (a BatchedQuadEnv
    other than the training env) every `eval_freq` vec-env steps and keeps a device copy of the best parameters and VecNormalize
    statistics by mean reward.  best_model_save_path: on every new best, also write `best_model.zip` there (QuadPPO.save: the
    parameters and Adam state of that evaluation) and, with VecNormalize, `best_model_vecnormalize.pkl` with its statistics.

    Unlike SB3, which evaluates in the middle of a rollout, the evaluation runs after the first train() that crosses a multiple of
    eval_freq: the collection is one replayed CUDA graph and is not split.  The callback flies its own MlpPolicyKernel over the
    training parameter blob (no output buffer, generator or Philox counter is shared with training, so training is unchanged) and
    reads the training VecNormalize observation statistics in place (sync_envs_normalization).  Single rank only."""

    def __init__(self, eval_env, eval_freq: int, n_eval_episodes: int = 10, deterministic: bool = True,
                 best_model_save_path: str | None = None):
        if int(eval_freq) < 1:
            raise ValueError("eval_freq must be >= 1")
        self.eval_env, self.eval_freq = eval_env, int(eval_freq)
        self.n_eval_episodes, self.deterministic = int(n_eval_episodes), bool(deterministic)
        self.best_model_save_path = best_model_save_path
        self.best_mean_reward = -math.inf
        self.last_mean_reward = -math.inf
        self.evaluations: list[dict] = []
        self._ppo = None
        self._best = None

    def init_callback(self, ppo) -> None:
        if self.eval_env is ppo.env:
            raise ValueError("EvalCallback: eval_env must not be the training env (evaluation resets it)")
        if ppo.world > 1:
            raise ValueError("EvalCallback is single-rank only: evaluate the shards with evaluate(..., n_global=...) instead")
        if self.eval_env.obs_dim != ppo.env.obs_dim or self.eval_env.device != ppo.env.device:
            raise ValueError("EvalCallback: eval_env differs from the training env in observation size or device")
        if self.best_model_save_path is not None:
            os.makedirs(self.best_model_save_path, exist_ok=True)
        if self._ppo is not ppo:
            impl = {v: k for k, v in IMPL.items()}[ppo.policy.impl]
            self.policy = MlpPolicyKernel(ppo.policy.state_dict, ppo.env.obs_dim, ppo.env.device, impl=impl)
            self.policy.params = ppo.policy.params
            self._ppo = ppo
            self._bucket = _vec_steps(ppo) // self.eval_freq

    def after_train(self, ppo) -> dict:
        """Called by QuadPPO.learn after every train(); returns the eval/* entries of the log when it evaluated, else {}."""
        due, self._bucket = _crossed(ppo, self.eval_freq, self._bucket)
        if not due:
            return {}
        vn = ppo.vecnorm
        res = evaluate(self.policy, self.eval_env, self.n_eval_episodes, self.deterministic, vecnorm=vn)
        rewards = res.episode_rewards()
        mean_reward, std_reward = float(np.mean(rewards)), float(np.std(rewards))
        out = {"eval/mean_reward": mean_reward, "eval/std_reward": std_reward,
               "eval/mean_ep_length": float(np.mean(res.episode_lengths())), "eval/success_rate": res.success_rate}
        self.evaluations.append(dict(out, timesteps=ppo.num_timesteps))
        self.last_mean_reward = mean_reward
        if mean_reward > self.best_mean_reward:
            self.best_mean_reward = mean_reward
            self._best = (ppo.policy.params.clone(), vn.obs_rms.stats.clone() if vn is not None else None,
                          vn.ret_rms.stats.clone() if vn is not None else None)
            if self.best_model_save_path is not None:
                path = self.best_model_save_path
                ppo.save(os.path.join(path, "best_model.zip"),
                         vecnormalize_path=os.path.join(path, "best_model_vecnormalize.pkl") if vn is not None else None)
        return out

    def best_state_dict(self) -> dict:
        """{"policy": SB3-named parameters of the best evaluation (feed to sb3_compat.save_policy_zip),
        "vecnorm": the DeviceVecNormalize.state_dict() fields at that evaluation, or None without VecNormalize}."""
        if self._best is None:
            raise RuntimeError("EvalCallback: no evaluation has run yet")
        params, obs_stats, ret_stats = self._best
        out = {"policy": unpack_params(params.cpu().numpy(), self._ppo.env.obs_dim), "vecnorm": None}
        vn = self._ppo.vecnorm
        if vn is not None:
            d = self._ppo.env.obs_dim
            sd = vn.state_dict()
            o, r = obs_stats.cpu().numpy(), ret_stats.cpu().numpy()
            sd.update(obs_mean=o[1:1 + d].copy(), obs_var=o[1 + d:].copy(), obs_count=float(o[0]),
                      ret_mean=float(r[1]), ret_var=float(r[2]), ret_count=float(r[0]))
            out["vecnorm"] = sd
        return out


class CheckpointCallback:
    """stable_baselines3 CheckpointCallback for QuadPPO.learn(callback=...): after the first train() that crosses each multiple of
    `save_freq` vec-env steps (EvalCallback's rule), writes `{name_prefix}_{num_timesteps}_steps.zip` (QuadPPO.save: every
    checkpoint resumes exactly with QuadPPO.load) and, with save_vecnormalize and a VecNormalize,
    `{name_prefix}_vecnormalize_{num_timesteps}_steps.pkl` into save_path.  template_zip is passed to QuadPPO.save.  Reads device
    state only, so training is unchanged.  Single rank (QuadPPO.save)."""

    def __init__(self, save_freq: int, save_path: str, name_prefix: str = "rl_model", save_vecnormalize: bool = False,
                 template_zip: str | None = None):
        if int(save_freq) < 1:
            raise ValueError("save_freq must be >= 1")
        self.save_freq, self.save_path, self.name_prefix = int(save_freq), save_path, name_prefix
        self.save_vecnormalize, self.template_zip = bool(save_vecnormalize), template_zip
        self._ppo = None

    def _path(self, kind: str, ext: str, steps: int) -> str:
        return os.path.join(self.save_path, f"{self.name_prefix}_{kind}{steps}_steps.{ext}")

    def init_callback(self, ppo) -> None:
        if ppo.world > 1:
            raise ValueError("CheckpointCallback is single-rank only")
        os.makedirs(self.save_path, exist_ok=True)
        if self._ppo is not ppo:
            self._ppo = ppo
            self._bucket = _vec_steps(ppo) // self.save_freq

    def after_train(self, ppo) -> dict:
        """Called by QuadPPO.learn after every train(); saves when due.  Adds nothing to the log."""
        due, self._bucket = _crossed(ppo, self.save_freq, self._bucket)
        if due:
            vn = ppo.vecnorm if self.save_vecnormalize else None
            ppo.save(self._path("", "zip", ppo.num_timesteps), template_zip=self.template_zip,
                     vecnormalize_path=self._path("vecnormalize_", "pkl", ppo.num_timesteps) if vn is not None else None)
        return {}
