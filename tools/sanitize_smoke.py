"""Small run of every kernel family at ragged sizes (partial warp tiles, partial 128-row policy tiles): a quick all-kernels
smoke, and the workload to put under compute-sanitizer (memcheck / racecheck) where that tool is available -- it is closed on the
build pool, so out-of-bounds protection here rests on the ragged-size parity tests against the oracle.
    python tools/sanitize_smoke.py"""
import os, sys
sys.path.insert(0, os.getcwd())
import torch
from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
from rl_aerial_manipulator_b200.pid import BatchedPID
from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
from rl_aerial_manipulator_b200.ppo import gae
from rl_aerial_manipulator_b200.vec_normalize import DeviceRunningMeanStd

n = 1000 + 13
g = torch.Generator(device="cuda").manual_seed(0)
for ver, prec, integ, kw in ((2, "f32", "rk4", {}), (1, "f32", "rk4", {}), (2, "f64", "rk4", {}), (2, "f64", "lsoda", {}),
                             (2, "f32", "rk4", {"v2_random_waypoints": True})):
    env = BatchedQuadEnv(n if integ == "rk4" else 77, env_version=ver, precision=prec, integrator=integ, seed=1, **kw)
    env.reset()
    rms = DeviceRunningMeanStd(env.obs_dim, "cuda")
    rms.attach(env, merge=True)
    for t in range(6):
        a = torch.rand((env.n_envs, 4), device="cuda", generator=g) * torch.tensor([0.5, 2, 2, 2], device="cuda") - torch.tensor([0, 1, 1, 1.0], device="cuda")
        out = env.step(a)
    env.fuse_obs_moments(None)
    if integ == "rk4":
        env.step_range(32, 200, a[32:232].contiguous())
    st = env.get_state()
    env.set_state(y=st["y"])
    pid = BatchedPID(env)
    pid.actions(None, 0.005)
    env.close()
for impl in ("fp32", "tensor", "tensor_fast"):
    pol = MlpPolicyKernel.from_npz("tests/golden/policy_v2.npz", device="cuda", impl=impl)
    obs = torch.randn((n, 20), device="cuda", generator=g)
    pol.forward(obs, torch.randn((n, 4), device="cuda", generator=g), norm_stats=rms.stats if False else None)
    stats = torch.zeros(41, dtype=torch.float64, device="cuda"); stats[0] = 1.0; stats[21:] = 1.0
    pol.forward(obs, None, norm_stats=stats, obs_norm_out=torch.empty_like(obs))
T = 8
r = torch.randn((T, n), device="cuda"); v = torch.randn((T, n), device="cuda")
s = (torch.rand((T, n), device="cuda") < 0.1).to(torch.uint8)
gae(r, v, s, torch.randn(n, device="cuda"), (torch.rand(n, device="cuda") < 0.1).to(torch.uint8), 0.995, 0.9)
# population kernels: K agents at a ragged n (qs_policy_forward_pop), one population minibatch update (qs_ppo_pop_update)
from rl_aerial_manipulator_b200.population import PopulationPPO
pop = PopulationPPO(BatchedQuadEnv(3 * 37, env_version=2, seed=1), 3, [0, 1, 2], n_steps=5, batch_size=100, n_epochs=1, rollout_graph=False)
pop.collect_rollouts()
pop.train()
pop.close()
torch.cuda.synchronize()
print("SANITIZE_SMOKE_DONE")
