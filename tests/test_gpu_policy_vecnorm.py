"""GPU tests of the VecNormalize and MlpPolicy kernels through the C-ABI, against the SB3 restatement
(oracle/sb3_oracle.py), a plain torch fp32 reference and the golden forward outputs (tests/golden/policy_*.npz)."""
import os

import numpy as np
import pytest
import torch

from oracle import sb3_oracle as so

pytestmark = pytest.mark.gpu


def t2n(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("tag,obs_dim", [("v2", 20), ("v1", 17)])
def test_policy_forward_matches_golden_and_torch(golden_dir, tag, obs_dim):
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    z = np.load(os.path.join(golden_dir, f"policy_{tag}.npz"))
    pol = MlpPolicyKernel.from_npz(os.path.join(golden_dir, f"policy_{tag}.npz"), device="cuda", impl="fp32")
    assert pol.obs_dim == obs_dim
    obs = torch.from_numpy(z["obs"]).cuda()
    a, v, lp = pol.forward(obs)                                   # deterministic: actions == mean
    # golden: torch CPU forward of the shipped SB3 weights; float32 kernel vs float64 truth, and vs float32 truth
    # tolerance: torch's own float32 forward is 3.9e-6 (means, |mu| <= 16) / 4e-4 (values, |V| <= 2048) away from
    # float64; the kernel's ex2.approx-based tanh adds ~1e-7 per activation -> 1e-4 / 5e-3 absolute
    np.testing.assert_allclose(t2n(a), z["mean_f64"], rtol=2e-5, atol=1e-4)
    np.testing.assert_allclose(t2n(v), z["value_f64"], rtol=2e-5, atol=5e-3)
    np.testing.assert_allclose(t2n(a), z["mean_f32"], rtol=2e-5, atol=1e-4)
    log_std = z["w.log_std"]
    np.testing.assert_allclose(t2n(lp), np.full(len(z["obs"]), -log_std.sum() - 2 * np.log(2 * np.pi)), rtol=1e-6)
    lo, hi = np.array([0, -1, -1, -1.0]), np.array([2, 1, 1, 1.0])
    np.testing.assert_array_equal(t2n(pol.actions_clipped), np.clip(t2n(a), lo, hi).astype(np.float32))


# stated tolerances per implementation: (|mean action| error, |value| error) against the float64 forward, for the shipped
# v2 policy (|mu| <= 16, |V| <= 2800).  torch's own float32 forward is (3.9e-6, 4e-4) away from float64.
#   fp32         CUDA-core FFMA, float32 throughout; ex2-based tanh                      measured (5e-6, 1.1e-3)
#   tensor       tcgen05, split-float16 operands (3 MMAs per k-step), float32 accumulate  measured (8e-6, 2.9e-3)
#   tensor_fast  tcgen05, single float16 operands, MUFU.TANH                              measured (1.7e-2, 4.5)
POLICY_TOL = {"fp32": (1e-4, 5e-3), "tensor": (1e-4, 1e-2), "tensor_fast": (6e-2, 20.0)}


@pytest.mark.parametrize("impl", ["fp32", "tensor", "tensor_fast"])
@pytest.mark.parametrize("n", [1, 63, 64, 65, 127, 129, 4099, 262144])
def test_policy_forward_stochastic_vs_oracle(golden_dir, n, impl):
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    pol = MlpPolicyKernel.from_npz(os.path.join(golden_dir, "policy_v2.npz"), device="cuda", impl=impl)
    tol_a, tol_v = POLICY_TOL[impl]
    g = torch.Generator(device="cuda").manual_seed(n)
    obs = torch.randn((n, 20), device="cuda", generator=g) * 0.7
    noise = torch.randn((n, 4), device="cuda", generator=g)
    a, v, lp = pol.forward(obs, noise)
    m = min(n, 4096)
    ao, vo, lpo, _ = so.mlp_policy_forward(pol.state_dict, t2n(obs[:m]), t2n(noise[:m]))
    np.testing.assert_allclose(t2n(a[:m]), ao, rtol=0, atol=tol_a)
    np.testing.assert_allclose(t2n(v[:m]), vo, rtol=0, atol=tol_v)
    np.testing.assert_allclose(t2n(lp[:m]), lpo, rtol=1e-5, atol=1e-5)
    # whole batch against the plain torch fp32 reference of the same op
    mean_t, value_t = so.torch_policy_forward(pol.state_dict, obs)
    a_t = mean_t + torch.exp(torch.from_numpy(pol.state_dict["log_std"]).cuda()) * noise
    assert (a - a_t).abs().max() < tol_a and (v - value_t).abs().max() < tol_v
    assert torch.equal(pol.actions_clipped, torch.minimum(torch.maximum(a, torch.tensor([0.0, -1, -1, -1], device="cuda")),
                                                          torch.tensor([2.0, 1, 1, 1], device="cuda")))


@pytest.mark.parametrize("impl", ["tensor", "tensor_fast"])
def test_policy_tensor_path_v1_weights(golden_dir, impl):
    """17-D observations (K padded 17 -> 32 inside the kernel) with the v1 4M policy."""
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    z = np.load(os.path.join(golden_dir, "policy_v1.npz"))
    pol = MlpPolicyKernel.from_npz(os.path.join(golden_dir, "policy_v1.npz"), device="cuda", impl=impl)
    tol_a, tol_v = POLICY_TOL[impl]
    a, v, _ = pol.forward(torch.from_numpy(z["obs"]).cuda())
    np.testing.assert_allclose(t2n(a), z["mean_f64"], rtol=0, atol=tol_a)
    np.testing.assert_allclose(t2n(v), z["value_f64"], rtol=0, atol=tol_v)


@pytest.mark.parametrize("impl", ["fp32", "tensor"])
def test_policy_forward_with_fused_vecnormalize(golden_dir, impl):
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    from rl_aerial_manipulator_b200.vec_normalize import DeviceRunningMeanStd
    pol = MlpPolicyKernel.from_npz(os.path.join(golden_dir, "policy_v2.npz"), device="cuda", impl=impl)
    n = 10000
    g = torch.Generator(device="cuda").manual_seed(1)
    obs = torch.randn((n, 20), device="cuda", generator=g) * 3 + 1
    obs[:, 6] = 1.0 - 1e-4 * torch.rand(n, device="cuda", generator=g)      # quaternion w near hover: mean ~1, std ~3e-5
    rms = DeviceRunningMeanStd(20, "cuda")
    rms.update(obs)
    normed = rms.normalize(obs)
    a1, v1, _ = pol.forward(normed)
    a1, v1 = a1.clone(), v1.clone()
    out = torch.empty_like(obs)
    a2, v2, _ = pol.forward(obs, norm_stats=rms.stats, obs_norm_out=out)
    # fp32: float64 normalisation like SB3; tensor: float32 hi/lo mean split, within 2 float32 ulp of it (|z| < 8 here)
    assert torch.allclose(out, normed, atol=1e-6 if impl == "fp32" else 2e-6)
    assert torch.allclose(a1, a2, atol=1e-4) and torch.allclose(v1, v2, atol=1e-2)


@pytest.mark.parametrize("d,n", [(20, 1 << 20), (17, 100003), (1, 65536), (20, 8), (20, 1)])
def test_batch_moments_and_running_update(d, n):
    from rl_aerial_manipulator_b200.vec_normalize import DeviceRunningMeanStd
    g = torch.Generator(device="cuda").manual_seed(d * 7 + n)
    rms = DeviceRunningMeanStd(d, "cuda")
    ref64 = so.RunningMeanStd((d,), dtype_batch=np.float64)
    ref32 = so.RunningMeanStd((d,), dtype_batch=np.float32)
    for it in range(3):
        x = torch.randn((n, d), device="cuda", generator=g) * (1 + it) + torch.arange(d, device="cuda") * 0.5
        x[:, 0] = 1.0 + 1e-4 * torch.randn(n, device="cuda", generator=g)       # a nearly constant column (quaternion w)
        m = t2n(rms.batch_moments(x))
        xn = t2n(x).astype(np.float64)
        assert m[0] == n
        np.testing.assert_allclose(m[1:1 + d], xn.mean(0), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(m[1 + d:], xn.var(0) * n, rtol=1e-9, atol=1e-12)
        rms.update(x)
        ref64.update(xn)
        ref32.update(t2n(x))
        s = t2n(rms.stats)
        assert abs(s[0] - ref64.count) < 1e-9
        np.testing.assert_allclose(s[1:1 + d], ref64.mean, rtol=1e-12, atol=1e-12)     # float64 restatement: exact arithmetic
        np.testing.assert_allclose(s[1 + d:], ref64.var, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(s[1:1 + d], ref32.mean, rtol=1e-4, atol=1e-4)      # SB3's float32 batch statistics
        np.testing.assert_allclose(s[1 + d:], ref32.var, rtol=1e-3, atol=1e-6)
        out = t2n(rms.normalize(x))
        want = np.clip((xn - ref64.mean) / np.sqrt(ref64.var + 1e-8), -10, 10)
        np.testing.assert_allclose(out, want, rtol=2e-5, atol=2e-5)


def test_device_vecnormalize_rollout_vs_oracle():
    """DeviceVecNormalize around the float64 env vs the SB3 restatement fed the same obs / rewards / dones."""
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    n = 512
    env = BatchedQuadEnv(n, env_version=1, precision="f64", integrator="rk4", obs_scaled=False, seed=3)   # rl_env.py + VecNormalize
    vn = DeviceVecNormalize(env, gamma=0.99)
    ref = so.VecNormalizeOracle(n, 17, gamma=0.99)
    obs = vn.reset()
    np.testing.assert_allclose(t2n(obs), ref.reset(t2n(env.obs)), rtol=2e-5, atol=2e-5)
    g = torch.Generator(device="cuda").manual_seed(0)
    for t in range(150):
        a = torch.rand((n, 4), device="cuda", generator=g) * torch.tensor([0.8, 2, 2, 2], device="cuda") - torch.tensor([0, 1, 1, 1.0], device="cuda")
        out = vn.step(a.float())
        want = ref.step(t2n(vn.raw_obs), t2n(out.reward), t2n(out.done))
        np.testing.assert_allclose(t2n(out.obs), want, rtol=3e-5, atol=3e-5)
    sd = vn.state_dict()
    np.testing.assert_allclose(sd["obs_mean"], ref.obs_rms.mean, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(sd["obs_var"], ref.obs_rms.var, rtol=1e-8, atol=1e-12)
    assert abs(sd["obs_count"] - ref.obs_rms.count) < 1e-6 and abs(sd["ret_count"] - ref.ret_rms.count) < 1e-6
    np.testing.assert_allclose(sd["ret_mean"], ref.ret_rms.mean, rtol=1e-5, atol=1e-5)      # returns are carried in float32 on the device
    np.testing.assert_allclose(sd["ret_var"], ref.ret_rms.var, rtol=1e-4)
    assert int(out.done.sum()) >= 0 and sd["obs_count"] > 151 * n


def test_vecnormalize_pkl_layout_roundtrip(golden_dir):
    """The reference's vec_normalize.pkl snapshot (17-D float64 mean/var, count 2031632.0001) loads into the device object."""
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    z = np.load(os.path.join(golden_dir, "vecnorm_v1.npz"))
    env = BatchedQuadEnv(64, env_version=1, precision="f32", obs_scaled=False)
    vn = DeviceVecNormalize(env, training=False)
    vn.load_state_dict({k: z[k] for k in z.files})
    sd = vn.state_dict()
    np.testing.assert_array_equal(sd["obs_mean"], z["obs_mean"])
    np.testing.assert_array_equal(sd["obs_var"], z["obs_var"])
    assert sd["obs_count"] == float(z["obs_count"]) == 2031632.0001 and sd["clip_obs"] == 10.0 and sd["gamma"] == 0.99
    obs = vn.reset()
    raw = t2n(env.obs).astype(np.float64)
    want = np.clip((raw - z["obs_mean"]) / np.sqrt(z["obs_var"] + 1e-8), -10, 10)
    np.testing.assert_allclose(t2n(obs), want, rtol=2e-5, atol=2e-5)
    assert float(vn.obs_rms.count) == 2031632.0001     # training=False: statistics frozen


@pytest.mark.parametrize("variant,precision,n", [("v2", "f32", 1 << 18), ("v2", "f64", 4099), ("v1", "f32", 33), ("v1", "f64", 70001)])
def test_fused_obs_moments_in_step_kernel(variant, precision, n):
    """qs_step_moments: the step kernel's own reduction of the observations it returns == qs_batch_moments(obs) == NumPy."""
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.vec_normalize import DeviceRunningMeanStd
    ver = 2 if variant == "v2" else 1
    env = BatchedQuadEnv(n, env_version=ver, precision=precision, seed=6)
    d = env.obs_dim
    fused = DeviceRunningMeanStd(d, "cuda")
    plain = DeviceRunningMeanStd(d, "cuda")
    env.reset()
    fused.attach(env)
    g = torch.Generator(device="cuda").manual_seed(2)
    for t in range(30):
        a = torch.rand((n, 4), device="cuda", generator=g) * torch.tensor([0.6, 2, 2, 2], device="cuda") - torch.tensor([0, 1, 1, 1.0], device="cuda")
        out = env.step(a.float())
        m_f = t2n(fused._moments).copy()
        m_p = t2n(plain.batch_moments(out.obs)).copy()
        x = t2n(out.obs).astype(np.float64)
        assert m_f[0] == n
        # the fused path adds 8 rows at a time in float32 around the running mean (SB3 itself takes the whole batch mean in
        # float32): 1e-6 of a standard deviation on the mean, 2e-6 relative on M2
        sd = x.std(0) + 1e-12
        assert np.all(np.abs(m_f[1:1 + d] - x.mean(0)) <= 1e-6 * sd + 1e-9)
        np.testing.assert_allclose(m_f[1 + d:], x.var(0) * n, rtol=2e-6, atol=1e-6)
        np.testing.assert_allclose(m_p[1:1 + d], x.mean(0), rtol=1e-12, atol=1e-12)
        fused.update_from_moments()
        plain.update(out.obs)
    np.testing.assert_allclose(t2n(fused.stats)[1:1 + d], t2n(plain.stats)[1:1 + d], rtol=0, atol=1e-6)
    np.testing.assert_allclose(t2n(fused.stats)[1 + d:], t2n(plain.stats)[1 + d:], rtol=3e-6, atol=1e-9)
    env.fuse_obs_moments(None)
    before = t2n(fused._moments).copy()
    env.step(a.float())
    np.testing.assert_array_equal(t2n(fused._moments), before)       # switched off: untouched
    env.close()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs on one node")
def test_peer_memory_moment_exchange_matches_nccl_two_ranks():
    """qs_xchg_merge (all-gather + Chan merge fused over NVLink peer memory) == NCCL all-gather + qs_vecnorm_merge, bit for bit,
    on every rank, eagerly and from a CUDA graph (tools/peer_exchange_check.py under torchrun)."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29517", os.path.join(root, "tools", "peer_exchange_check.py")], cwd=root, capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and "PEER_EXCHANGE_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])


@pytest.mark.gpu
def test_peer_memory_moment_exchange_two_processes_one_device():
    """The same exchange kernel between two PROCESSES on one GPU (CUDA IPC works on the same device; NCCL does not, so the checker is
    oracle/sb3_oracle.merge_moments and the rendezvous gloo): runs on a single-GPU box, where the two-rank test above is skipped."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29531", os.path.join(root, "tools", "peer_exchange_one_device.py")], cwd=root, capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and "PEER_ONE_DEVICE_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-6000:])


@pytest.mark.gpu
def test_step_kernel_merges_running_statistics_itself():
    """attach(env, merge=True): RunningMeanStd.update happens inside qs_step (the kernel that finishes the moments); the running
    statistics must equal, bit for bit, those of the two-launch path (moments triplet -> qs_vecnorm_merge) on the same env."""
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.vec_normalize import DeviceRunningMeanStd
    stats = {}
    for merge in (False, True):
        env = BatchedQuadEnv(20000, env_version=2, precision="f32", seed=9)
        rms = DeviceRunningMeanStd(env.obs_dim, "cuda")
        env.reset()
        rms.attach(env, merge=merge)
        g = torch.Generator(device="cuda").manual_seed(4)
        for t in range(25):
            a = torch.rand((20000, 4), device="cuda", generator=g) * torch.tensor([1.0, 2, 2, 2], device="cuda") - torch.tensor([0, 1, 1, 1.0], device="cuda")
            env.step(a)
            rms.update_from_moments()                      # no-op when the env merges
        stats[merge] = t2n(rms.stats).copy()
        assert abs(stats[merge][0] - (1e-4 + 25 * 20000)) < 1e-6
        env.close()
    np.testing.assert_array_equal(stats[True], stats[False])
