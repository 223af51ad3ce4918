"""PPO pieces (rl-aerial-manipulator_b200/ppo.py, csrc/qs_gae.cu) against NumPy restatements of SB3 2.6.0."""
import math
import os

import numpy as np
import pytest
import torch


def sb3_gae(rewards, values, episode_starts, last_values, dones, gamma, lam):
    """RolloutBuffer.compute_returns_and_advantage, restated."""
    T = rewards.shape[0]
    adv = np.zeros_like(rewards)
    last = 0.0
    for step in reversed(range(T)):
        if step == T - 1:
            nnt, nv = 1.0 - dones.astype(np.float32), last_values
        else:
            nnt, nv = 1.0 - episode_starts[step + 1], values[step + 1]
        delta = rewards[step] + gamma * nv * nnt - values[step]
        last = delta + gamma * lam * nnt * last
        adv[step] = last
    return adv, adv + values


def random_minibatch(rng, B, D, sd):
    """A synthetic minibatch with every loss branch populated: ratios inside and on both sides of the clip range, both signs of the
    advantage."""
    from oracle import ppo_oracle as po
    obs = rng.standard_normal((B, D)).astype(np.float32)
    act = (rng.standard_normal((B, 4)) * 1.5).astype(np.float32)
    adv = (rng.standard_normal(B) * 3 + 1).astype(np.float32)
    ret = (rng.standard_normal(B) * 10).astype(np.float32)
    net = po.make_torch_actor_critic(sd, D, torch.float64)
    with torch.no_grad():
        _, lp, _ = net.evaluate_actions(torch.from_numpy(obs).double(), torch.from_numpy(act).double())
    oldlp = (lp.numpy() + 0.3 * rng.standard_normal(B)).astype(np.float32)
    return obs, act, oldlp, adv, ret


def perturbed_state_dict(D, seed):
    """SB3 initialisation + noise, so that biases, log_std and the small action head all carry gradient-relevant values."""
    from rl_aerial_manipulator_b200.ppo import init_state_dict
    rng = np.random.default_rng(seed)
    return {k: (np.asarray(v, np.float32) + 0.05 * rng.standard_normal(np.shape(v)).astype(np.float32)) for k, v in init_state_dict(D, seed).items()}


def test_numpy_ppo_update_matches_torch_autograd():
    """The hand-derived NumPy backward / clipping / Adam of oracle/ppo_oracle.py against torch autograd + clip_grad_norm_ +
    torch.optim.Adam(eps=1e-5) in float64: ten consecutive updates, parameters equal to rounding."""
    from oracle import ppo_oracle as po
    rng = np.random.default_rng(0)
    for D, B in ((20, 128), (17, 37)):
        sd = {k: v.astype(np.float64) for k, v in perturbed_state_dict(D, 3).items()}
        net = po.make_torch_actor_critic(sd, D, torch.float64)
        opt = torch.optim.Adam(net.parameters(), lr=2e-4, eps=1e-5)
        st, sdn = po.adam_init(sd), {k: v.copy() for k, v in sd.items()}
        for it in range(10):
            batch = tuple(np.asarray(x, np.float64) for x in random_minibatch(rng, B, D, {k: v for k, v in sdn.items()}))
            s = po.update(sdn, st, batch, lr=2e-4, ent_coef=0.01)
            t = po.torch_update(net, opt, tuple(torch.from_numpy(x) for x in batch), ent_coef=0.01)
            assert abs(s["loss"] - t[0]) < 1e-10 * max(1, abs(t[0])) and abs(s["grad_norm"] - t[4]) < 1e-10 * max(1, t[4])
        err = max(np.abs(sdn[k] - v.detach().numpy()).max() for k, v in net.state_dict().items())
        assert err < 1e-12, err


def f64_state_dict(D, seed):
    return {k: v.astype(np.float64) for k, v in perturbed_state_dict(D, seed).items()}


@pytest.mark.parametrize("normalize_advantage", [True, False])
@pytest.mark.parametrize("case", ["random", "one_row", "constant_advantage"])
def test_numpy_minibatch_stats_and_grads_match_torch_autograd(case, normalize_advantage):
    """minibatch_grads against torch autograd in float64 for both advantage settings, including SB3's two diagnostics
    (clip_fraction, approx_kl) and the edges of the normalisation: a one-row minibatch (SB3 skips the normalisation, since
    torch.std of one element is NaN) and constant advantages (std 0: (A - mean) / (0 + 1e-8) = 0)."""
    from oracle import ppo_oracle as po
    D, B = 20, {"random": 37, "one_row": 1, "constant_advantage": 64}[case]
    rng = np.random.default_rng(B)
    sd = f64_state_dict(D, 4)
    batch = [np.asarray(x, np.float64) for x in random_minibatch(rng, B, D, sd)]
    if case == "constant_advantage":
        batch[3][:] = np.float32(1.7)             # a float32 buffer value: its mean is exact in float64, so A - mean = 0 exactly
    hp = dict(clip_range=0.15, ent_coef=0.01, vf_coef=0.7, normalize_advantage=normalize_advantage)
    stats, grads = po.minibatch_grads(sd, *batch, **hp)
    net = po.make_torch_actor_critic(sd, D, torch.float64)
    opt = torch.optim.SGD(net.parameters(), lr=0.0)
    t = po.torch_update(net, opt, tuple(torch.from_numpy(x) for x in batch), max_grad_norm=1e30, **hp)   # coef 1: unclipped
    for i, k in enumerate(("loss", "policy_gradient_loss", "value_loss", "entropy_loss")):
        assert math.isfinite(stats[k]) and abs(stats[k] - t[i]) <= 1e-12 * max(1.0, abs(t[i])), (k, stats[k], t[i])
    assert abs(stats["clip_fraction"] - t[5]) < 1e-7                    # SB3 takes the mean of a float32 mask
    assert abs(stats["approx_kl"] - t[6]) <= 1e-12 * max(1.0, abs(t[6]))
    for name, p in net.named_parameters():
        np.testing.assert_allclose(grads[name], p.grad.numpy(), rtol=1e-10, atol=1e-13, err_msg=name)
    if case == "random":
        assert 0.0 < stats["clip_fraction"] < 1.0 and stats["approx_kl"] > 0.0        # both sides of the clip range populated
    if case == "constant_advantage" and normalize_advantage:
        assert stats["policy_gradient_loss"] == 0.0 and not grads["action_net.weight"].any()


def test_numpy_update_passes_betas_and_eps_to_adam():
    """update(betas=, eps=) reaches adam_step: six updates against torch.optim.Adam with the same non-default betas / eps / lr
    and a clipping max_grad_norm, float64, parameters and both moments equal to rounding."""
    from oracle import ppo_oracle as po
    D, B = 17, 50
    rng = np.random.default_rng(6)
    sd = f64_state_dict(D, 8)
    hp = dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.3)
    net = po.make_torch_actor_critic(sd, D, torch.float64)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, betas=(0.8, 0.95), eps=1e-7)
    st = po.adam_init(sd)
    for it in range(6):
        batch = tuple(np.asarray(x, np.float64) for x in random_minibatch(rng, B, D, sd))
        s = po.update(sd, st, batch, lr=1e-3, betas=(0.8, 0.95), eps=1e-7, **hp)
        t = po.torch_update(net, opt, tuple(torch.from_numpy(x) for x in batch), **hp)
        assert abs(s["grad_norm"] - t[4]) < 1e-10 * t[4] and t[4] > hp["max_grad_norm"] and s["batch_size"] == B
    for name, p in net.named_parameters():
        np.testing.assert_allclose(sd[name], p.detach().numpy(), rtol=0, atol=1e-12, err_msg=name)
        np.testing.assert_allclose(st["m"][name], opt.state[p]["exp_avg"].numpy(), rtol=1e-9, atol=1e-15, err_msg=name)
        np.testing.assert_allclose(st["v"][name], opt.state[p]["exp_avg_sq"].numpy(), rtol=1e-9, atol=1e-18, err_msg=name)
    assert st["step"] == 6 == int(opt.state[next(net.parameters())]["step"])


@pytest.mark.parametrize("batch_size", [32, 23, 100])
def test_numpy_train_pass_matches_torch_training_loop(batch_size):
    """train_pass (PPO.train restated: n_epochs over given permutations, minibatches cut as RolloutBuffer.get cuts them) against
    the same loop over torch_update in float64.  70 rows: batch 32 leaves a ragged 6-row minibatch, 23 a one-row one, 100 (larger
    than the buffer) one minibatch of all rows per epoch."""
    from oracle import ppo_oracle as po
    D, total, n_epochs = 20, 70, 3
    rng = np.random.default_rng(batch_size)
    sd = f64_state_dict(D, 9)
    buffers = tuple(np.asarray(x, np.float64) for x in random_minibatch(rng, total, D, sd))
    perms = [rng.permutation(total) for _ in range(n_epochs)]
    hp = dict(lr=3e-4, clip_range=0.2, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5)
    net = po.make_torch_actor_critic(sd, D, torch.float64)
    opt = torch.optim.Adam(net.parameters(), lr=hp["lr"], eps=1e-5)
    st = po.adam_init(sd)
    stats = po.train_pass(sd, st, buffers, perms, batch_size, **hp)
    sizes = [len(i) for i in po.minibatches(perms[0], batch_size)]
    assert sum(sizes) == total and sizes[:-1] == [min(batch_size, total)] * (len(sizes) - 1)
    assert len(stats) == n_epochs * len(sizes) == st["step"] and [s["batch_size"] for s in stats[-len(sizes):]] == sizes
    tb = tuple(torch.from_numpy(x) for x in buffers)
    k = 0
    for perm in perms:
        for idx in po.minibatches(perm, batch_size):
            t = po.torch_update(net, opt, tuple(x[torch.from_numpy(idx)] for x in tb), **{k_: v for k_, v in hp.items() if k_ != "lr"})
            for i, key in enumerate(("loss", "policy_gradient_loss", "value_loss", "entropy_loss", "grad_norm", "clip_fraction", "approx_kl")):
                tol = 1e-7 if key == "clip_fraction" else 1e-10 * max(1.0, abs(t[i]))      # SB3: mean of a float32 mask
                assert abs(stats[k][key] - t[i]) <= tol, (k, key, stats[k][key], t[i])
            k += 1
    for name, p in net.named_parameters():
        np.testing.assert_allclose(sd[name], p.detach().numpy(), rtol=0, atol=1e-12, err_msg=name)


def test_init_and_packing_roundtrip():
    from rl_aerial_manipulator_b200.policy import pack_params, unpack_params
    from rl_aerial_manipulator_b200.ppo import init_state_dict
    for D in (17, 20):
        sd = init_state_dict(D, seed=3)
        assert sd["action_net.weight"].shape == (4, 64) and np.allclose(sd["log_std"], 0)
        w = sd["mlp_extractor.policy_net.2.weight"]
        np.testing.assert_allclose(w @ w.T, 2 * np.eye(64), atol=1e-4)       # orthogonal rows, gain sqrt(2)
        w = sd["action_net.weight"]
        np.testing.assert_allclose(w @ w.T, 1e-4 * np.eye(4), atol=1e-8)
        blob = pack_params(sd, D)
        back = unpack_params(blob, D)
        assert set(back) == set(sd) and all(np.array_equal(back[k], sd[k]) for k in sd)


@pytest.mark.gpu
def test_gae_kernel_vs_sb3_restatement():
    from rl_aerial_manipulator_b200.ppo import gae
    rng = np.random.default_rng(1)
    for T, n in ((1, 7), (16, 1000), (64, 4099)):
        rewards = rng.normal(size=(T, n)).astype(np.float32) * 10
        values = rng.normal(size=(T, n)).astype(np.float32) * 50
        starts = (rng.random((T, n)) < 0.1).astype(np.uint8)
        last_values = rng.normal(size=n).astype(np.float32) * 50
        dones = (rng.random(n) < 0.1).astype(np.uint8)
        c = lambda a: torch.from_numpy(a).cuda()
        adv, ret = gae(c(rewards), c(values), c(starts), c(last_values), c(dones), 0.995, 0.9)
        a_np, r_np = sb3_gae(rewards.astype(np.float64), values.astype(np.float64), starts.astype(np.float64), last_values.astype(np.float64),
                             dones, 0.995, 0.9)
        np.testing.assert_allclose(adv.cpu().numpy(), a_np, rtol=1e-4, atol=1e-3)
        np.testing.assert_allclose(ret.cpu().numpy(), r_np, rtol=1e-4, atol=1e-3)


# T, n, gamma, lambda, P(episode start), P(last done)
GAE_EDGES = {
    "reference_shape": (2048, 8, 0.995, 0.9, 0.01, 0.1),          # v1/rl_train_vecN.py: 8 envs x n_steps 2048
    "undiscounted": (2048, 8, 1.0, 1.0, 0.002, 0.0),                # gamma = lambda = 1: advantages sum rewards over whole episodes
    "every_step_a_start": (64, 1000, 0.995, 0.9, 1.0, 0.1),
    "all_last_dones": (64, 1000, 0.995, 0.9, 0.05, 1.0),
    "one_env": (300, 1, 0.995, 0.9, 0.01, 1.0),
    "ragged_block": (50, 257, 0.995, 0.9, 0.1, 0.5),               # 256-thread blocks: one env in a second block
}
# the kernel is SB3's float32 recurrence: each of the T steps adds a few roundings of its operands, which accumulate like a
# random walk.  Bound: sqrt(T) * 2^-24 * (max|rewards| + max|values| + max|advantages|); worst measured on an NVIDIA B200 (1000 W
# power limit): 0.18 of it (gamma = lambda = 1, T = 2048).


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(GAE_EDGES))
def test_gae_kernel_edges_vs_sb3_restatement(case):
    """qs_gae at the reference's own shape, gamma = lambda = 1, episode starts at every step, every env done at the end, one env
    and a ragged last block, against the float64 restatement within a bound that grows with sqrt(T)."""
    from rl_aerial_manipulator_b200.ppo import gae
    T, n, gamma, lam, p_start, p_done = GAE_EDGES[case]
    rng = np.random.default_rng(T + n)
    rewards = (rng.normal(size=(T, n)) * 10).astype(np.float32)
    values = (rng.normal(size=(T, n)) * 50).astype(np.float32)
    starts = (rng.random((T, n)) < p_start).astype(np.uint8)
    last_values = (rng.normal(size=n) * 50).astype(np.float32)
    dones = (rng.random(n) < p_done).astype(np.uint8)
    c = lambda a: torch.from_numpy(a).cuda()
    adv, ret = gae(c(rewards), c(values), c(starts), c(last_values), c(dones), gamma, lam)
    a_np, r_np = sb3_gae(rewards.astype(np.float64), values.astype(np.float64), starts.astype(np.float64), last_values.astype(np.float64),
                         dones, gamma, lam)
    if p_start == 1.0:                       # every next step is a new episode: delta without bootstrap, no carried advantage
        np.testing.assert_allclose(a_np[:-1], rewards[:-1].astype(np.float64) - values[:-1], rtol=0, atol=1e-12)
    scale = np.abs(rewards).max() + np.abs(values).max() + np.abs(a_np).max()
    bound = np.sqrt(T) * 2.0 ** -24 * scale
    err_a, err_r = np.abs(adv.cpu().numpy() - a_np).max(), np.abs(ret.cpu().numpy() - r_np).max()
    print(f"measured gae {case}: {err_a / bound:.4f} {err_r / bound:.4f} of the bound {bound:.3g}")
    assert err_a <= bound and err_r <= bound, (err_a, err_r, bound)


PPO_HP = dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("D,B", [(20, 128), (17, 128), (20, 37), (20, 1000), (20, 16384)])
def test_ppo_update_kernel_gradient_vs_oracle(D, B):
    """qs_ppo_grad (one launch: gather, forward, loss, backward, fixed-order reduction) against the float64 NumPy restatement of
    PPO.train's loss and its hand-derived gradient (pinned to torch autograd on the CPU): every parameter gradient, the loss terms."""
    from oracle import ppo_oracle as po
    from rl_aerial_manipulator_b200.policy import pack_params
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel
    rng = np.random.default_rng(B + D)
    sd = perturbed_state_dict(D, 7)
    total = 3 * B + 5
    obs, act, oldlp, adv, ret = random_minibatch(rng, total, D, sd)
    idx = rng.permutation(total)[:B].astype(np.int64)
    c = lambda a: torch.from_numpy(a).cuda()
    params = c(pack_params(sd, D))
    opt = PpoUpdateKernel(params, D, learning_rate=2e-4, **PPO_HP)
    g = opt.gradient(c(obs), c(act), c(oldlp), c(adv), c(ret), c(idx)).cpu().numpy()
    stats_k = opt.read_stats()
    stats, grads = po.minibatch_grads(sd, obs[idx], act[idx], oldlp[idx], adv[idx], ret[idx], **{k: PPO_HP[k] for k in ("clip_range", "ent_coef", "vf_coef")})
    want = pack_params({k: np.asarray(v, np.float32) for k, v in grads.items()}, D)
    scale = np.abs(want).max()
    assert np.abs(g - want).max() < 2e-5 * scale, (np.abs(g - want).max(), scale)
    for k in ("loss", "policy_gradient_loss", "value_loss", "entropy_loss"):
        assert abs(stats_k[k] - stats[k]) < 2e-5 * max(1.0, abs(stats[k])), (k, stats_k[k], stats[k])
    assert abs(stats_k["grad_norm"] - np.sqrt(sum((v ** 2).sum() for v in grads.values()))) < 1e-4 * scale * 100
    assert stats_k["batch_size"] == B
    assert torch.equal(params, c(pack_params(sd, D)))          # qs_ppo_grad leaves the parameters alone
    opt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("B", [128, 300])
def test_ppo_update_kernel_ten_updates_vs_torch_autograd_and_oracle(B):
    """Ten consecutive minibatch updates by qs_ppo_update (hand-written forward/backward/clip/Adam) against (i) the update the way
    SB3 computes it -- torch modules + autograd + clip_grad_norm_ + torch.optim.Adam(eps=1e-5), float32 on the same GPU -- and
    (ii) the float64 NumPy oracle: parameters within 1e-5 after ten steps (VERDICT r01 item 7's bar), Adam state included."""
    from oracle import ppo_oracle as po
    from rl_aerial_manipulator_b200.policy import pack_params
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel
    D = 20
    rng = np.random.default_rng(B)
    sd = perturbed_state_dict(D, 11)
    c = lambda a: torch.from_numpy(a).cuda()
    params = c(pack_params(sd, D))
    opt = PpoUpdateKernel(params, D, learning_rate=2e-4, **PPO_HP)
    net = po.make_torch_actor_critic(sd, D).cuda()
    topt = torch.optim.Adam(net.parameters(), lr=2e-4, eps=1e-5)
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    st64 = po.adam_init(sd64)
    for it in range(10):
        batch = random_minibatch(rng, B, D, {k: v for k, v in sd64.items()})
        opt.update(*(c(x) for x in batch))
        t = po.torch_update(net, topt, tuple(c(x) for x in batch), **PPO_HP)
        s = po.update(sd64, st64, tuple(np.asarray(x, np.float64) for x in batch), lr=2e-4, **PPO_HP)
        k = opt.read_stats()
        assert abs(k["loss"] - s["loss"]) < 1e-4 * max(1.0, abs(s["loss"])) and abs(k["grad_norm"] - s["grad_norm"]) < 1e-4 * max(1.0, s["grad_norm"])
        assert abs(k["loss"] - t[0]) < 1e-4 * max(1.0, abs(t[0]))
    got = params.cpu().numpy()
    want_t = pack_params({k: v.detach().cpu().numpy() for k, v in net.state_dict().items()}, D)
    want_o = pack_params({k: v.astype(np.float32) for k, v in sd64.items()}, D)
    assert np.abs(got - want_o).max() < 1e-5, np.abs(got - want_o).max()
    assert np.abs(got - want_t).max() < 1e-5, np.abs(got - want_t).max()
    m, v, step = opt.adam_state()
    assert int(step.item()) == 10
    m_o = pack_params({k: a.astype(np.float32) for k, a in st64["m"].items()}, D)
    assert np.abs(m.cpu().numpy() - m_o).max() < 1e-5 * max(1.0, np.abs(m_o).max())
    opt.close()


@pytest.mark.gpu
def test_ppo_update_kernel_is_deterministic_and_grid_independent():
    """Fixed reduction order: the same minibatch gives bit-identical gradients run to run; rows 0..B-1 without an index list equal
    the same rows through idx."""
    from rl_aerial_manipulator_b200.policy import pack_params
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel
    D, B = 20, 5000
    rng = np.random.default_rng(2)
    sd = perturbed_state_dict(D, 5)
    batch = [torch.from_numpy(x).cuda() for x in random_minibatch(rng, B, D, sd)]
    params = torch.from_numpy(pack_params(sd, D)).cuda()
    opt = PpoUpdateKernel(params, D, **PPO_HP)
    g0 = opt.gradient(*batch).clone()
    g1 = opt.gradient(*batch).clone()
    g2 = opt.gradient(*batch, torch.arange(B, device="cuda")).clone()
    assert torch.equal(g0, g1) and torch.equal(g0, g2)
    opt.close()


@pytest.mark.gpu
def test_quad_ppo_iterations_run_and_parameters_move():
    """Two collect/train iterations on 4096 envs with VecNormalize (ragged last minibatch included): finite losses, parameters move,
    rollout bookkeeping is consistent, the rollout kernel reads the updated blob."""
    from oracle import sb3_oracle as so
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    n = 4096
    env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=1)
    vn = DeviceVecNormalize(env, norm_obs=True, norm_reward=True, gamma=0.995)
    ppo = QuadPPO(env, vecnorm=vn, n_steps=32, batch_size=50000, n_epochs=3, policy_impl="fp32", seed=0)    # 131072 = 2 x 50000 + 31072
    before = ppo.policy.params.clone()
    logs = []
    ppo.learn(2 * 32 * n, log=logs.append)
    assert len(logs) == 2 and all(math.isfinite(l[k]) for l in logs for k in ("loss", "policy_gradient_loss", "value_loss", "entropy_loss"))
    assert logs[-1]["batch_size"] == 31072 and ppo.num_timesteps == 2 * 32 * n
    assert int(ppo.opt.adam_state()[2].item()) == 2 * 3 * 3
    after = ppo.policy.params
    assert float((after - before).abs().max()) > 1e-5 and bool(torch.isfinite(after).all())
    assert abs(float(vn.obs_rms.count) - (1e-4 + n * (1 + 2 * 32))) < 1e-3          # reset + every step
    assert float(ppo.rewards.abs().max()) <= 10.0 + 0.995 * float(ppo.values.abs().max()) + 1e-3   # norm_reward: clipped at clip_reward (+ bootstrap)
    # GAE bookkeeping: returns = advantages + values
    assert torch.allclose(ppo.returns, ppo.advantages + ppo.values, atol=1e-3)
    obs = ppo.obs[5].contiguous()
    mean_t, v_t = so.torch_policy_forward(ppo.state_dict(), obs)
    a_k, v_k, _ = ppo.policy.forward(obs)
    assert float((v_k - v_t).abs().max()) < 5e-3 and float((a_k - mean_t).abs().max()) < 1e-4
    env.close()


@pytest.mark.gpu
def test_quad_ppo_reference_hyperparameters_small_run():
    """The reference's own settings (v1/rl_train_vecN.py: 8 envs, n_steps 2048, batch 128, 10 epochs): one iteration = 1280 kernel
    launches; two runs with the same seed are bit-identical (deterministic reductions, device-side RNG streams)."""
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    params = []
    for rep in range(2):
        env = BatchedQuadEnv(8, env_version=1, precision="f32", seed=3)
        ppo = QuadPPO(env, n_steps=256, batch_size=128, n_epochs=4, policy_impl="fp32", seed=5)
        logs = []
        ppo.learn(2 * 256 * 8, log=logs.append)
        assert len(logs) == 2 and all(math.isfinite(v) for l in logs for k, v in l.items() if k.endswith("loss"))
        params.append(ppo.policy.params.clone())
        env.close()
    assert torch.equal(params[0], params[1])


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs on one node")
def test_ppo_two_ranks_stay_in_lockstep():
    """BASELINE configs[4] mechanics on 2 ranks (tools/ppo_multi_rank_check.py under torchrun): sharded envs, VecNormalize statistics
    through the peer-memory exchange, NCCL gradient all-reduce -> bit-identical parameters and statistics on every rank."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29523", os.path.join(root, "tools", "ppo_multi_rank_check.py")], cwd=root, capture_output=True,
                       text=True, timeout=400)
    assert r.returncode == 0 and "PPO_MULTI_RANK_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])


@pytest.mark.gpu
def test_ppo_two_processes_one_device_stay_in_lockstep():
    """The same check with both ranks on ONE GPU (gloo rendezvous; the moment exchange still runs over CUDA IPC peer memory, the
    gradient all-reduce through gloo): sharded envs + qs_ppo_grad / all-reduce / qs_ppo_apply keep parameters and statistics
    bit-identical on both ranks.  Runs on the single-GPU box where the two-GPU test is skipped."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, QS_ONE_DEVICE="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", os.path.join(root, "tools", "ppo_multi_rank_check.py")], cwd=root, capture_output=True,
                       text=True, timeout=600, env=env)
    assert r.returncode == 0 and "PPO_MULTI_RANK_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])


@pytest.mark.gpu
def test_collect_rollouts_bookkeeping_vs_sb3_restatement():
    """OnPolicyAlgorithm.collect_rollouts semantics of QuadPPO.collect_rollouts, replayed on a twin env and recomputed in NumPy:
    the stored (unclipped) actions clipped to the box drive the env; rewards[t] = env reward + gamma * V(terminal_observation) for
    envs that hit the time limit only (TimeLimit.truncated), untouched otherwise; episode_starts[t] = dones of the previous step
    (ones at the start); values[t] = V(obs[t]); advantages / returns = SB3's GAE over those buffers with V(last obs), last dones."""
    from oracle import sb3_oracle as so
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    n, T, gamma, lam = 384, 8, 0.995, 0.9
    envs = []
    for _ in range(2):
        e = BatchedQuadEnv(n, env_version=2, precision="f32", seed=21)
        e.reset()
        st = e.get_state()
        st["current_step"][: n // 3] = torch.arange(n // 3, device="cuda", dtype=torch.int32) % 6 + 1994   # truncate within the rollout (limit 2000)
        st["y"][n // 3: n // 2, 2] = 0.13                                                             # and some crash (terminated)
        st["y"][n // 3: n // 2, 5] = -4.0
        e.set_state(**st)
        envs.append(e)
    env, twin = envs
    ppo = QuadPPO(env, n_steps=T, batch_size=n * T, n_epochs=1, gamma=gamma, gae_lambda=lam, policy_impl="fp32", seed=3)
    ppo._last_obs = env.obs                                  # start from the injected state instead of a fresh reset
    obs0 = env.obs.clone()
    ppo.collect_rollouts()
    sd = ppo.state_dict()
    V = lambda o: so.torch_policy_forward(sd, o)[1]
    lo = torch.tensor([0.0, -1, -1, -1], device="cuda")
    hi = torch.tensor([2.0, 1, 1, 1], device="cuda")
    obs = obs0
    prev_done = np.ones(n, np.uint8)
    rew, starts, n_trunc, n_term = np.zeros((T, n)), np.zeros((T, n), np.uint8), 0, 0
    for t in range(T):
        assert torch.equal(ppo.obs[t], obs)
        torch.testing.assert_close(ppo.values[t], V(obs), rtol=0, atol=5e-3)
        out = twin.step(torch.minimum(torch.maximum(ppo.actions[t], lo), hi).contiguous())
        flags = out.flags.cpu().numpy()
        r = out.reward.double().cpu().numpy().copy()
        trunc_only = (flags & 3) == 2
        if trunc_only.any():
            tv = V(out.terminal_obs[torch.from_numpy(trunc_only).cuda()]).double().cpu().numpy()
            r[trunc_only] += gamma * tv
        n_trunc += int(trunc_only.sum())
        n_term += int(((flags & 1) != 0).sum())
        rew[t], starts[t] = r, prev_done
        prev_done = ((flags & 3) != 0).astype(np.uint8)
        obs = out.obs.clone()
    assert n_trunc >= n // 6 and n_term >= n // 12            # both kinds of episode end happened
    np.testing.assert_array_equal(ppo.episode_starts.cpu().numpy(), starts)
    np.testing.assert_allclose(ppo.rewards.cpu().numpy(), rew, rtol=1e-5, atol=5e-3)
    last_v = V(obs).double().cpu().numpy()
    a_np, r_np = sb3_gae(rew, ppo.values.double().cpu().numpy(), starts.astype(np.float64), last_v, prev_done, gamma, lam)
    np.testing.assert_allclose(ppo.advantages.cpu().numpy(), a_np, rtol=1e-4, atol=2e-2)
    np.testing.assert_allclose(ppo.returns.cpu().numpy(), r_np, rtol=1e-4, atol=2e-2)
    env.close()
    twin.close()


@pytest.mark.gpu
def test_graph_replayed_collection_equals_eager_collection():
    """QuadPPO(rollout_graph=True) replays ONE captured collection step (fixed addresses, rollout-buffer slot from a device counter);
    it must fill the rollout buffers exactly as the eager loop does -- same kernels, same order, same random stream -- over two
    collections (the second one is replays only), with VecNormalize (norm_obs + norm_reward) in the loop and envs that hit the time
    limit or crash inside the rollout."""
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    n, T = 512, 12
    runs = []
    for use_graph in (False, True):
        env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=11)
        env.reset()
        st = env.get_state()
        st["current_step"][: n // 4] = torch.arange(n // 4, device="cuda", dtype=torch.int32) % 9 + 1990      # truncations inside the rollouts
        st["y"][n // 4: n // 3, 2] = 0.13
        st["y"][n // 4: n // 3, 5] = -4.0                                                               # and crashes
        env.set_state(**st)
        vn = DeviceVecNormalize(env, norm_obs=True, norm_reward=True, gamma=0.995)
        ppo = QuadPPO(env, vecnorm=vn, n_steps=T, batch_size=n * T, n_epochs=1, policy_impl="fp32", seed=4, rollout_graph=use_graph)
        ppo._last_obs = env.obs
        vn.obs_rms.update(env.obs)
        vn.obs_rms.attach(env, merge=True)
        snaps = []
        for _ in range(2):
            ppo.collect_rollouts()
            snaps.append({k: getattr(ppo, k).clone() for k in ("obs", "actions", "values", "logp", "rewards", "episode_starts", "advantages", "returns")})
            snaps[-1]["stats"] = vn.obs_rms.stats.clone()
            snaps[-1]["ret_stats"] = vn.ret_rms.stats.clone()
            snaps[-1]["ep"] = torch.tensor([ppo.ep_count, ppo.num_timesteps])
        assert (ppo._graph is not None) == use_graph
        runs.append(snaps)
        env.close()
    for a, b in zip(*runs):
        for k in a:
            assert torch.equal(a[k], b[k]), k
    assert int(runs[0][0]["ep"][0]) > 0                              # episodes did end (time limit, crash) inside the first rollout


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
def test_rollout_record_kernels_vs_numpy(f64):
    """qs_rollout_record_pre / _post against a NumPy restatement of RolloutBuffer.add + the reward bookkeeping of collect_rollouts
    (reward normalisation in float32, gamma * V(terminal obs) for TimeLimit.truncated envs only, last dones, episode statistics),
    float32 and float64 env outputs, ragged n, slot t taken from device memory and advanced by the post kernel."""
    import ctypes as C
    from rl_aerial_manipulator_b200 import ppo as ppo_mod
    from rl_aerial_manipulator_b200._cabi import load_library
    lib = load_library()
    ppo_mod._bind(lib)
    rng = np.random.default_rng(3)
    n, d, T = 1000 + 37, 20, 5
    dev = "cuda"
    real = np.float64 if f64 else np.float32
    t_dev = torch.tensor([2], dtype=torch.int64, device=dev)
    bufs = {k: torch.full(shp, -7.0, dtype=torch.float32, device=dev) for k, shp in
            (("obs", (T, n, d)), ("act", (T, n, 4)), ("val", (T, n)), ("logp", (T, n)), ("rew", (T, n)))}
    starts = torch.full((T, n), 9, dtype=torch.uint8, device=dev)
    last_dones = torch.from_numpy(rng.integers(0, 2, n).astype(np.uint8)).to(dev)
    obs, act = rng.standard_normal((n, d)).astype(np.float32), rng.standard_normal((n, 4)).astype(np.float32)
    val, logp = rng.standard_normal(n).astype(np.float32), rng.standard_normal(n).astype(np.float32)
    g = lambda a: torch.from_numpy(a).to(dev)
    p = lambda x: C.c_void_p(x.data_ptr())
    d_obs, d_act, d_val, d_logp = g(obs), g(act), g(val), g(logp)
    ld0 = last_dones.cpu().numpy().copy()
    assert lib.qs_rollout_record_pre(p(t_dev), n, d, p(d_obs), p(d_act), p(d_val), p(d_logp), p(last_dones), p(bufs["obs"]), p(bufs["act"]),
                                     p(bufs["val"]), p(bufs["logp"]), p(starts), None) == 0
    reward = (rng.standard_normal(n) * 30).astype(real)
    flags = rng.choice(np.array([0, 0, 0, 1, 2, 3, 0x12, 0x21], np.uint8), n)
    ep_ret = (rng.standard_normal(n) * 1000).astype(real)
    tv = (rng.standard_normal(n) * 50).astype(np.float32)
    ret_stats = torch.tensor([100.0, 3.0, 412.7], dtype=torch.float64, device=dev)
    ep_stats = torch.tensor([5.5, 2.0], dtype=torch.float64, device=dev)
    ws = torch.zeros(2 * 1024 + 1, dtype=torch.float64, device=dev)
    gamma, eps, clip = 0.995, 1e-8, 10.0
    d_rew, d_flags, d_ep, d_tv = g(reward), g(flags), g(ep_ret), g(tv)
    for use_norm in (True, False):
        t_before = int(t_dev.item())
        assert lib.qs_rollout_record_post(p(t_dev), n, p(d_rew), int(f64), p(d_flags), p(d_ep), p(d_tv), gamma,
                                          C.c_void_p(ret_stats.data_ptr() + 16) if use_norm else None, eps, clip, p(bufs["rew"]), p(last_dones),
                                          p(ep_stats), p(ws), None) == 0
        torch.cuda.synchronize()
        r = reward.astype(np.float32)
        if use_norm:
            r = np.clip(r / np.float32(np.sqrt(412.7 + eps)), np.float32(-clip), np.float32(clip))
        f3 = flags & 3
        r = np.where(f3 == 2, r + np.float32(gamma) * tv, r).astype(np.float32)
        np.testing.assert_array_equal(bufs["rew"][t_before].cpu().numpy(), r)
        assert int(t_dev.item()) == t_before + 1
    np.testing.assert_array_equal(last_dones.cpu().numpy(), (f3 != 0).astype(np.uint8))
    want = np.array([5.5 + 2 * ep_ret[f3 != 0].astype(np.float64).sum(), 2.0 + 2 * (f3 != 0).sum()])
    np.testing.assert_allclose(ep_stats.cpu().numpy(), want, rtol=1e-12)
    for k, a in (("obs", obs), ("act", act), ("val", val), ("logp", logp)):
        np.testing.assert_array_equal(bufs[k][2].cpu().numpy(), a)
        assert float(bufs[k][1].max()) == -7.0 and float(bufs[k][3].min()) == -7.0          # the neighbouring slots are untouched
    np.testing.assert_array_equal(starts[2].cpu().numpy(), ld0)
    assert int(starts[1].min()) == 9 and float(bufs["rew"][4].max()) == -7.0
