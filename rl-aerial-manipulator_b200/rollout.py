"""FusedRollout -- one kernel launch per rollout step (`qs_rollout_step`, csrc/qs_rollout.cu): VecNormalize normalisation ->
MlpPolicy forward on tcgen05 -> Gaussian sampling / log-prob / clipping -> env step -> auto-reset -> VecNormalize moments.

Replaces one iteration of stable_baselines3 `OnPolicyAlgorithm.collect_rollouts` over the reference's vec env (call sites
initial-implementation-v2/rl_train.py:27-56, initial-implementation-v1/rl_train_vecN.py:10-36): `policy(obs)` -> `np.clip` ->
`VecNormalize.step_wait` / `DummyVecEnv.step_wait` -> `WaypointQuadEnv.step` for every env of the shard.  The separate calls
(`MlpPolicyKernel.forward` + `BatchedQuadEnv.step`) stay available and produce the same numbers; this is the throughput path.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _cabi
from ._cabi import QsRolloutArgs, check
from .batched_env import BatchedQuadEnv, StepOut
from .policy import ACTION_HIGH, ACTION_LOW, NACT, MlpPolicyKernel


class FusedRollout:
    """env: a float32 / RK4 BatchedQuadEnv (already reset).  policy: MlpPolicyKernel (its parameter blob is converted to the
    tensor-core operand image here; call `refresh_policy()` after the parameters change).  vecnorm: DeviceRunningMeanStd attached
    to `env` (its statistics normalise the observations and are updated from the moments the kernel reduces), or None.

    sample: "mean" (deterministic), "philox" (noise drawn in the kernel: Philox4x32-10 keyed on `noise_seed`, counter = global env
    id and a device-resident step counter, so CUDA-graph replays draw fresh noise and shards draw what the whole batch would), or
    "noise" (pass a float32[n,4] standard-normal tensor to step())."""

    def __init__(self, env: BatchedQuadEnv, policy: MlpPolicyKernel, vecnorm=None, sample: str = "philox", noise_seed: int = 0,
                 store_obs_norm: bool = False, norm_eps: float = 1e-8, norm_clip: float = 10.0):
        if env.precision != "f32" or env.integrator != "rk4":
            raise ValueError("FusedRollout needs a float32 / RK4 env")
        if getattr(env, "dynamics_randomization", None) is not None:
            raise ValueError("FusedRollout: the fused rollout kernel has no dynamics randomisation; step the env with a policy "
                             "forward + env.step (QuadPPO does), or disarm it")
        self.env, self.policy, self.vecnorm = env, policy, vecnorm
        self.lib = env.lib
        self.mode = {"mean": _cabi.SAMPLE_MEAN, "noise": _cabi.SAMPLE_NOISE, "philox": _cabi.SAMPLE_PHILOX}[sample]
        dev, n, d = env.device, env.n_envs, env.obs_dim
        self.image = torch.empty(int(self.lib.qs_policy_image_bytes()), dtype=torch.uint8, device=dev)
        self.noise_step = torch.zeros(1, dtype=torch.int64, device=dev)
        self.noise_seed = int(noise_seed)
        self.actions = torch.empty((n, NACT), dtype=torch.float32, device=dev)
        self.actions_clipped = torch.empty((n, NACT), dtype=torch.float32, device=dev)
        self.values = torch.empty(n, dtype=torch.float32, device=dev)
        self.logp = torch.empty(n, dtype=torch.float32, device=dev)
        self.obs_norm = torch.empty((n, d), dtype=torch.float32, device=dev) if store_obs_norm else None
        self.norm_eps, self.norm_clip = float(norm_eps), float(norm_clip)
        self.refresh_policy()

    def refresh_policy(self) -> None:
        """Rebuild the operand image from `policy.params` (after an optimiser step)."""
        rc = self.lib.qs_policy_prepare(C.c_void_p(self.policy.params.data_ptr()), self.env.obs_dim, C.c_void_p(self.image.data_ptr()),
                                        C.c_void_p(torch.cuda.current_stream(self.env.device).cuda_stream))
        check(self.lib, None, rc, "qs_policy_prepare")

    def step(self, noise: torch.Tensor | None = None, out_actions=None, out_values=None, out_logp=None, out_obs_norm=None) -> StepOut:
        """One rollout step from `env.obs`.  Afterwards: `actions` (sampled, unclipped), `actions_clipped`, `values`, `logp` hold the
        policy's outputs for the PRE-step observations, the returned StepOut (env buffers) the env's results, `env.obs` the next
        observations.  out_*: write the rollout-buffer rows straight into the caller's tensors (e.g. slices of a [T, n, ...] buffer)."""
        env = self.env
        a = QsRolloutArgs()
        p = lambda t: t.data_ptr() if t is not None else None
        a.policy_image = p(self.image)
        a.obs = p(env.obs)
        a.norm_stats = p(self.vecnorm.stats) if self.vecnorm is not None else None
        a.norm_eps, a.norm_clip = self.norm_eps, self.norm_clip
        a.sample_mode = self.mode
        if self.mode == _cabi.SAMPLE_NOISE:
            if noise is None or noise.dtype != torch.float32 or tuple(noise.shape) != (env.n_envs, NACT) or not noise.is_contiguous():
                raise ValueError("sample='noise' needs a contiguous float32[n,4] noise tensor")
            a.noise = p(noise)
        a.noise_seed = self.noise_seed
        a.noise_step = p(self.noise_step)
        a.clip_lo[:] = ACTION_LOW
        a.clip_hi[:] = ACTION_HIGH
        obs_norm = out_obs_norm if out_obs_norm is not None else self.obs_norm
        a.obs_norm_out = p(obs_norm)
        a.actions_out = p(out_actions if out_actions is not None else self.actions)
        a.actions_clipped_out = p(self.actions_clipped)
        a.values_out = p(out_values if out_values is not None else self.values)
        a.logp_out = p(out_logp if out_logp is not None else self.logp)
        a.obs_next = p(env.obs)
        a.reward_out, a.flags_out = p(env.reward), p(env.flags)
        a.terminal_obs_out, a.ep_return_out, a.ep_len_out = p(env.terminal_obs), p(env.ep_return), p(env.ep_len)
        check(self.lib, env._h, self.lib.qs_rollout_step(env._h, C.byref(a), env._stream()), "qs_rollout_step")
        return StepOut(env.obs, env.reward, env.flags, env.terminal_obs, env.ep_return, env.ep_len)

    def status(self) -> int:
        """0, or the code of an internal hand-over that timed out (synchronises the device)."""
        return int(self.lib.qs_rollout_status())
