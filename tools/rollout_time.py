"""Timing of the rollout step variants on one B200 (CUDA events around CUDA-graph replays, 1,048,576 envs by default):
policy forward alone (pipeline kernel), separate-launch rollout step, fused rollout step.
    python tools/rollout_time.py [n_envs] [steps]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv  # noqa: E402
from rl_aerial_manipulator_b200.policy import MlpPolicyKernel  # noqa: E402
from rl_aerial_manipulator_b200.rollout import FusedRollout  # noqa: E402
from rl_aerial_manipulator_b200.vec_normalize import DeviceRunningMeanStd  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 100
NPZ = os.path.join(ROOT, "tests", "golden", "policy_v2.npz")


def timed(fn, reps=steps, unroll=4):
    for _ in range(8):
        fn()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(unroll):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps // unroll):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (reps // unroll * unroll)


env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=0)
env.reset()
rms = DeviceRunningMeanStd(20, "cuda")
rms.update(env.obs)
rms.attach(env, merge=True)
gen = torch.Generator(device="cuda").manual_seed(0)
noise = torch.randn((n, 4), device="cuda", generator=gen)
res = {}
pol = MlpPolicyKernel.from_npz(NPZ, device="cuda", impl="tensor_pipeline")
res["policy"] = timed(lambda: pol.forward(env.obs, noise))
res["policy + vecnorm"] = timed(lambda: pol.forward(env.obs, noise, norm_stats=rms.stats))


def separate():
    pol.forward(env.obs, noise, norm_stats=rms.stats)
    env.step(pol.actions_clipped)


res["separate rollout step"] = timed(separate)
for sample in ("noise", "philox"):
    fused = FusedRollout(env, pol, vecnorm=rms, sample=sample)
    res[f"fused rollout step ({sample})"] = timed((lambda: fused.step(noise)) if sample == "noise" else (lambda: fused.step()))
    assert fused.status() == 0, fused.status()
fused = FusedRollout(env, pol, vecnorm=rms, sample="philox", store_obs_norm=True)
res["fused rollout step (philox, obs_norm stored)"] = timed(lambda: fused.step())
for k, v in res.items():
    print(f"{k:55s} {v * 1e3:9.1f} us   {n / v / 1e6:8.1f} M env-steps/s")
