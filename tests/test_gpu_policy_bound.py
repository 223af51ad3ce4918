"""GPU tests: every policy-forward entry point against the float64 oracle under the propagated error bound of
tests/policy_bound.py, on the generated weight sets (not only the shipped ones) -- qs_policy_forward for every impl, the in-kernel
Philox forward at the bench's shape, the fused rollout step's operand image (qs_policy_prepare), QuadPPO's default `auto` policy
(the tcgen05 kernel from 16,384 envs on) and its compacted time-limit bootstrap above 65,536 envs.  Each check prints
max(err / bound)."""
import numpy as np
import pytest
import torch

import policy_bound as pb
from test_gpu_rollout import philox_normal_oracle

pytestmark = pytest.mark.gpu

LO, HI = np.array([0.0, -1, -1, -1]), np.array([2.0, 1, 1, 1])
t2n = lambda t: t.detach().cpu().numpy()


def sample_rows(n, k=8192, seed=0):
    """all rows up to k; else the first and last 128-row tiles and a fixed random sample."""
    if n <= k:
        return np.arange(n)
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([np.arange(128), np.arange(n - 128, n), rng.choice(n, k - 256, replace=False)]))


def within(tag, got_mean, got_value, sd, obs, impl, norm=None, e0=None, eps=None):
    """mean / value rows against the oracle under the bound; prints and returns max(err / bound).  eps: the mean was recovered as
    actions - exp(log_std) eps, so the bound widens by that recovery's float32 rounding (see check_definitions)."""
    m, v, bm, bv = pb.forward_with_bound(sd, obs, impl, norm, e0=e0)
    if eps is not None:
        ls = np.abs(np.asarray(sd["log_std"], np.float64))
        bm = bm + 2.0 ** -23 * (np.abs(got_mean) + 2 * np.exp(ls) * np.abs(eps)) + (3 + 1.2 * ls) * 2.0 ** -23 * np.exp(ls) * np.abs(eps)
    rm, rv = pb.max_ratio(got_mean, got_value, m, v, bm, bv)
    print(f"{tag}: max(err/bound) mean {rm:.3g} value {rv:.3g}")
    assert rm <= 1.0 and rv <= 1.0, (tag, rm, rv)
    return max(rm, rv)


def std_of(sd):
    return np.exp(np.asarray(sd["log_std"], np.float64))


def check_definitions(sd, mean_k, eps, a, ac, lp):
    """actions = mean + exp(log_std) eps to float32 rounding (exp by __expf: (3 + 1.2 |log_std|) ulp), logp as SB3 computes it,
    actions_clipped = clip(actions) exactly."""
    ls = np.asarray(sd["log_std"], np.float64)
    std = np.exp(ls)
    tol = 2.0 ** -23 * (np.abs(a) + np.abs(mean_k)) + (3 + 1.2 * np.abs(ls)) * 2.0 ** -23 * std * np.abs(eps)
    assert (np.abs(a - (mean_k + std * eps)) <= tol).all()
    lp_o = np.sum(-0.5 * eps ** 2 - ls - 0.5 * np.log(2 * np.pi), axis=1)
    np.testing.assert_allclose(lp, lp_o, rtol=2e-6, atol=2e-6 * (1 + np.abs(ls).sum()))
    assert np.array_equal(ac, np.minimum(np.maximum(a, LO.astype(np.float32)), HI.astype(np.float32)))


def batch(D, n, seed):
    ins = pb.input_sets(D, rows=1024, seed=seed)
    raw = np.concatenate([x for k, (x, st) in ins.items() if st is None])
    x, st = ins["vecnorm"]
    return np.resize(raw, (n, D)), np.resize(x, (n, D)), st


SIZES = [1, 127, 128, 129, 16383, 16384, 148 * 128 * 2 + 77, 262144]


@pytest.mark.parametrize("impl,sizes", [("fp32", SIZES), ("tensor", SIZES), ("tensor_fast", SIZES), ("auto", [16383, 16384])])
def test_policy_forward_within_bound(golden_dir, impl, sizes):
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    worst = {}
    for D in (20, 17):
        for wi, (wn, sd) in enumerate(pb.weight_sets(golden_dir, D).items()):
            pol = MlpPolicyKernel(sd, D, "cuda", impl=impl)
            for n in (sizes if wn == "shipped" else [sizes[(wi + D) % len(sizes)]]):
                bimpl = impl if impl != "auto" else ("tensor" if n >= 16384 else "fp32")
                raw, xn, st = batch(D, n, seed=n)
                rows = sample_rows(n)
                g = torch.Generator(device="cuda").manual_seed(n)
                noise = torch.randn((n, 4), device="cuda", generator=g)
                # without normalisation, deterministic and with noise
                obs = torch.from_numpy(raw).cuda()
                a0, v0, _ = pol.forward(obs)
                mean_k, v0 = t2n(a0)[rows].astype(np.float64), t2n(v0)[rows]
                r = within(f"{impl} obs_dim={D} {wn} n={n}", mean_k, v0, sd, raw[rows], bimpl)
                a, v, lp = pol.forward(obs, noise)
                a, v, lp, ac = t2n(a), t2n(v), t2n(lp), t2n(pol.actions_clipped)
                assert np.array_equal(v[rows], v0)
                check_definitions(sd, mean_k, t2n(noise)[rows].astype(np.float64), a[rows].astype(np.float64), ac[rows], lp[rows])
                a2, v2, _ = pol.forward(obs, noise)
                assert np.array_equal(t2n(a2), a) and np.array_equal(t2n(v2), v), "second launch differs"
                # with VecNormalize statistics, with and without obs_norm_out
                obs = torch.from_numpy(xn).cuda()
                stats = torch.from_numpy(st).cuda()
                out = torch.full((n, D), float("nan"), device="cuda")
                a1, v1, _ = pol.forward(obs, noise, norm_stats=stats, obs_norm_out=out)
                a1, v1 = t2n(a1).copy(), t2n(v1).copy()
                mean_n = a1[rows] - std_of(sd) * t2n(noise)[rows]
                r = max(r, within(f"{impl} obs_dim={D} {wn} n={n} vecnorm", mean_n, v1[rows], sd, xn[rows], bimpl, st, eps=t2n(noise)[rows]))
                vn, e0 = pb.normalised_input(xn[rows], bimpl if bimpl != "fp32" else "fp32", st)
                assert (np.abs(t2n(out)[rows] - vn) <= e0).all(), "obs_norm_out outside e_0"
                a3, v3, _ = pol.forward(obs, noise, norm_stats=stats)
                assert np.array_equal(t2n(a3), a1) and np.array_equal(t2n(v3), v1)
                worst[(D, wn)] = max(worst.get((D, wn), 0.0), r)
    for (D, wn), r in worst.items():
        print(f"SUMMARY qs_policy_forward impl={impl} obs_dim={D} {wn}: max(err/bound) = {r:.3g}")


def test_forward_sampled_bench_shape(golden_dir):
    """qs_policy_forward_philox at 1,048,576 envs with VecNormalize statistics and env_id_offset = 2^33 (the bench's step)."""
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    n, D, seed, off = 1 << 20, 20, 0x0123456789ABCDEF, 1 << 33
    for wn in ("shipped", "trained_like", "wide_range"):
        sd = pb.weight_sets(golden_dir, D)[wn]
        pol = MlpPolicyKernel(sd, D, "cuda", impl="tensor")
        _, xn, st = batch(D, n, seed=7)
        obs, stats = torch.from_numpy(xn).cuda(), torch.from_numpy(st).cuda()
        mean = t2n(pol.forward(obs, norm_stats=stats)[0]).astype(np.float64)
        out = torch.empty((n, D), device="cuda")
        a, v, lp = pol.forward_sampled(obs, noise_seed=seed, env_id_offset=off, norm_stats=stats, obs_norm_out=out)
        rows = sample_rows(n, 65536, seed=1)
        a, v, lp, ac = t2n(a)[rows].astype(np.float64), t2n(v)[rows], t2n(lp)[rows], t2n(pol.actions_clipped)[rows]
        eps = philox_normal_oracle(seed, off + rows.astype(np.uint64), 0)
        std = std_of(sd)
        # device __sincosf / __log2f against NumPy, and the float32 rounding of the actions divided by std
        err = np.abs((a - mean[rows]) / std - eps)
        assert (err <= 2e-4 * (1 + np.abs(eps)) + 2.0 ** -22 * (np.abs(a) + np.abs(mean[rows])) / std).all(), err.max()
        within(f"forward_sampled 1M {wn}", mean[rows], v, sd, xn[rows], "tensor", st)
        assert np.array_equal(ac, np.minimum(np.maximum(a.astype(np.float32), LO.astype(np.float32)), HI.astype(np.float32)))
        ls = np.asarray(sd["log_std"], np.float64)
        np.testing.assert_allclose(lp, np.sum(-0.5 * eps ** 2 - ls - 0.5 * np.log(2 * np.pi), axis=1), rtol=1e-4, atol=1e-4)
        vn, e0 = pb.normalised_input(xn[rows], "tensor", st)
        assert (np.abs(t2n(out)[rows] - vn) <= e0).all()
        assert pol.lib.qs_rollout_status() == 0


@pytest.mark.parametrize("sample", ["noise", "mean"])
def test_fused_rollout_policy_outputs_and_refresh(golden_dir, sample):
    """FusedRollout reads the operand image qs_policy_prepare builds: its policy outputs are within the bound, and after the
    parameters change they follow the old weights until refresh_policy() and the new ones after it."""
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel, pack_params
    from rl_aerial_manipulator_b200.rollout import FusedRollout
    n, D = 148 * 128 + 5, 20
    ws = pb.weight_sets(golden_dir, D)
    old, new = ws["init_perturbed"], ws["wide_range"]
    env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=5)
    env.reset()
    pol = MlpPolicyKernel(old, D, "cuda", impl="tensor")
    fused = FusedRollout(env, pol, sample=sample)
    g = torch.Generator(device="cuda").manual_seed(3)

    def step(sd, tag):
        obs = t2n(env.obs).copy()
        noise = torch.randn((n, 4), device="cuda", generator=g) if sample == "noise" else None
        fused.step(noise)
        assert fused.status() == 0
        eps = t2n(noise).astype(np.float64) if noise is not None else np.zeros((n, 4))
        a, v = t2n(fused.actions).astype(np.float64), t2n(fused.values)
        within(f"fused sample={sample} {tag}", a - std_of(sd) * eps, v, sd, obs, "tensor", eps=eps)
        return obs, a, v, eps
    step(old, "init_perturbed")
    pol.params.copy_(torch.from_numpy(pack_params(new, D)).cuda())
    obs, a, v, eps = step(old, "init_perturbed after a parameter change, before refresh_policy()")
    m, vv, bm, bv = pb.forward_with_bound(new, obs, "tensor")
    assert (np.abs(v - vv) > bv).any(), "the new weights were used before refresh_policy()"
    fused.refresh_policy()
    step(new, "wide_range after refresh_policy()")
    env.close()


def _twins(n, seed, truncate, crash):
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    envs = []
    for _ in range(2):
        e = BatchedQuadEnv(n, env_version=2, precision="f32", seed=seed)
        e.reset()
        st = e.get_state()
        st["current_step"][truncate] = (torch.arange(n, device="cuda", dtype=torch.int32)[truncate] % 4) + 1996   # time limit 2000
        st["y"][crash, 2] = 0.13
        st["y"][crash, 5] = -4.0
        e.set_state(**st)
        envs.append(e)
    return envs


def test_quadppo_auto_policy_on_the_tensor_path(golden_dir):
    """QuadPPO(policy_impl="auto") at 16,384 envs runs the tcgen05 kernel: values[t] on the stored (kernel-normalised) obs[t], and
    every time-limit bootstrap and last-value forward (through _aux), against the oracle with the collecting weights; after train()
    the next forward uses the updated blob.  VecNormalize with norm_obs and norm_reward, two iterations."""
    from rl_aerial_manipulator_b200.policy import unpack_params
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    n, T, D = 16384, 8, 20
    env, _ = _twins(n, 3, slice(0, n // 4), slice(n // 4, n // 3))
    vn = DeviceVecNormalize(env, norm_obs=True, norm_reward=True, gamma=0.995)
    ppo = QuadPPO(env, vecnorm=vn, n_steps=T, batch_size=n * T // 4, n_epochs=1, seed=2, policy_impl="auto", rollout_graph=False)
    ppo._last_obs = env.obs
    vn.obs_rms.update(env.obs)
    vn.obs_rms.attach(env, merge=True)
    calls = []
    aux_forward = ppo._aux.forward

    def spy(obs, noise=None, norm_stats=None, **kw):
        stats = None if norm_stats is None else t2n(norm_stats).copy()
        out = aux_forward(obs, noise, norm_stats=norm_stats, **kw)
        calls.append((t2n(obs).copy(), stats, t2n(out[1]).copy()))
        return out
    ppo._aux.forward = spy
    for it in range(2):
        calls.clear()
        ppo.collect_rollouts()
        sd = unpack_params(t2n(ppo.policy.params), D)
        worst = 0.0
        for t in range(T):
            m, v, bm, bv = pb.forward_with_bound(sd, t2n(ppo.obs[t]), "tensor", e0=0.0)
            worst = max(worst, float((np.abs(t2n(ppo.values[t]) - v) / bv).max()))
        print(f"QuadPPO auto it={it} values[t]: max(err/bound) = {worst:.3g}")
        assert worst <= 1.0
        assert len(calls) == T + 1                                  # T bootstrap forwards (every env's terminal_obs) + last values
        worst = 0.0
        for k, (obs, stats, vals) in enumerate(calls):
            rows = sample_rows(len(obs), 4096, seed=k)
            _, v, _, bv = pb.forward_with_bound(sd, obs[rows], "tensor", stats)
            worst = max(worst, float((np.abs(vals[rows] - v) / bv).max()))
        print(f"QuadPPO auto it={it} _aux (bootstrap, last values): max(err/bound) = {worst:.3g}")
        assert worst <= 1.0
        ppo.train()
        sd_new = unpack_params(t2n(ppo.policy.params), D)
        assert not np.array_equal(sd_new["value_net.weight"], sd["value_net.weight"])
        x = t2n(ppo.obs[0])
        a, v, _ = ppo.policy.forward(ppo.obs[0].contiguous())
        within(f"QuadPPO auto it={it} after train()", t2n(a).astype(np.float64), t2n(v), sd_new, x, "tensor", e0=0.0)
    env.close()


@pytest.mark.parametrize("rollout_graph", [False, True])
def test_compacted_bootstrap_vs_sb3(golden_dir, rollout_graph):
    """Above 65,536 envs the time-limit bootstrap compacts the truncated envs into _boot_cap slots.  On a twin env driven by the
    stored actions: an env that was only truncated gets reward = normalised env reward + gamma V(normalised terminal obs) within
    gamma * bound; every other env's reward is left as is.  VecNormalize frozen (training=False) so the normalisation is a fixed
    function the test can restate."""
    from rl_aerial_manipulator_b200.policy import unpack_params
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    n, T, D, gamma = 131072, 6, 20, 0.995
    env, twin = _twins(n, 4, slice(0, n // 5), slice(n // 5, n // 4))
    vn = DeviceVecNormalize(env, norm_obs=True, norm_reward=True, gamma=gamma, training=False)
    vn.obs_rms.update(env.obs)
    vn.ret_rms.stats[2] = 4.0                                          # ret var
    ppo = QuadPPO(env, vecnorm=vn, n_steps=T, batch_size=n, n_epochs=1, gamma=gamma, seed=1, policy_impl="auto", rollout_graph=rollout_graph)
    assert ppo._boot_cap == 65536 < n
    ppo._last_obs = env.obs
    ppo.collect_rollouts()
    assert (ppo._graph is not None) == rollout_graph
    sd = unpack_params(t2n(ppo.policy.params), D)
    st = t2n(vn.obs_rms.stats)
    worst, n_trunc, n_term = 0.0, 0, 0
    for t in range(T):
        out = twin.step(torch.minimum(torch.maximum(ppo.actions[t], torch.tensor(LO, dtype=torch.float32, device="cuda")),
                                      torch.tensor(HI, dtype=torch.float32, device="cuda")).contiguous())
        flags = t2n(out.flags)
        if t + 1 < T:
            assert np.array_equal(t2n(ppo.episode_starts[t + 1]), ((flags & 3) != 0).astype(np.uint8))
        r_norm = t2n(torch.clamp(out.reward / torch.sqrt(vn.ret_rms.var[0] + vn.epsilon), -vn.clip_reward, vn.clip_reward))   # as SB3 / QuadPPO
        got = t2n(ppo.rewards[t])
        tr = (flags & 3) == 2
        assert np.array_equal(got[~tr], r_norm[~tr])
        if tr.any():
            _, v, _, bv = pb.forward_with_bound(sd, t2n(out.terminal_obs)[tr], "tensor", st, eps=vn.epsilon, clip=vn.clip_obs)
            want = r_norm[tr].astype(np.float64) + gamma * v
            err = np.abs(got[tr] - want)
            bound = gamma * bv + 2.0 ** -23 * np.abs(want)
            assert (err <= bound).all(), (t, (err / bound).max())
            worst = max(worst, float((err / bound).max()))
        n_trunc += int(tr.sum())
        n_term += int(((flags & 1) != 0).sum())
    assert n_trunc >= n // 6 and n_term >= n // 30
    print(f"compacted bootstrap rollout_graph={rollout_graph}: {n_trunc} truncations, max(err/bound) = {worst:.3g}")
    env.close()
    twin.close()


def test_boot_cap_overflow():
    """With boot_cap lowered: exactly `cap` truncations in one step is fine, `cap + 1` raises the documented RuntimeError."""
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    n, cap = 4096, 64
    for k, raises in ((cap, False), (cap + 1, True)):
        from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
        env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=8)
        env.reset()
        st = env.get_state()
        st["current_step"][:k] = 1999
        env.set_state(**st)
        ppo = QuadPPO(env, n_steps=6, batch_size=n * 6, n_epochs=1, seed=1, policy_impl="auto", boot_cap=cap, rollout_graph=False)
        ppo._last_obs = env.obs
        if raises:
            with pytest.raises(RuntimeError, match=f"more than {cap} envs hit the time limit"):
                ppo.collect_rollouts()
        else:
            ppo.collect_rollouts()
            assert bool((ppo.episode_starts[1:, :k] != 0).any(0).all())      # all k ended inside the rollout, none raised
        env.close()
