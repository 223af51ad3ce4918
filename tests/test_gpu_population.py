"""PopulationPPO on the B200: the two population kernels against their solo counterparts, and K agents trained in the same
launches against K solo QuadPPO runs, bit for bit (parameters, Adam state, rollout buffers, env state, statistics)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SEEDS = [0, 7, 42, 123]
HYPER = dict(learning_rate=[2e-4, 3e-4, 1e-4, 5e-4], ent_coef=[0.01, 0.0005, 0.0001, 0.0], clip_range=[0.2, 0.1, 0.3, 0.25],
             vf_coef=[0.5, 0.25, 1.0, 0.75], max_grad_norm=[0.5, 0.3, 1.0, 0.7], normalize_advantage=[True, False, True, False])


def _perturbed_blob(d, seed):
    from rl_aerial_manipulator_b200.policy import pack_params
    from rl_aerial_manipulator_b200.ppo import init_state_dict
    rng = np.random.default_rng(seed)
    sd = init_state_dict(d, seed)
    return pack_params({k: np.asarray(v, np.float32) + 0.05 * rng.standard_normal(np.shape(v)).astype(np.float32) for k, v in sd.items()}, d)


@pytest.mark.parametrize("K,B,d", [(1, 1, 20), (1, 128, 20), (3, 1000, 20), (3, 128, 17), (8, 128, 20), (8, 65536, 20),
                                   (3, 1, 17), (8, 1000, 17), (3, 65536, 17), (1, 65536, 20), (8, 1, 20), (1, 1000, 17)])
def test_population_update_equals_solo_updates(K, B, d):
    import ctypes as C
    from rl_aerial_manipulator_b200._cabi import QsPpoHyper, load_library
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel, STAT_KEYS
    lib = load_library()
    dev = torch.device("cuda", 0)
    R = max(2 * B, 4096)
    g = torch.Generator(device=dev).manual_seed(K * 1000 + B)
    obs = torch.randn((R, d), device=dev, generator=g)
    act = torch.randn((R, 4), device=dev, generator=g)
    oldlp = torch.randn(R, device=dev, generator=g) - 5
    adv = torch.randn(R, device=dev, generator=g)
    ret = torch.randn(R, device=dev, generator=g) * 10
    blobs = torch.from_numpy(np.stack([_perturbed_blob(d, 11 + a) for a in range(K)])).to(dev)
    hp = {k: (v * 3)[:K] for k, v in HYPER.items()}
    solo = [PpoUpdateKernel(blobs[a].clone(), d, clip_range=hp["clip_range"][a], ent_coef=hp["ent_coef"][a], vf_coef=hp["vf_coef"][a],
                            max_grad_norm=hp["max_grad_norm"][a], learning_rate=hp["learning_rate"][a],
                            normalize_advantage=hp["normalize_advantage"][a]) for a in range(K)]
    params = blobs.clone()
    h = C.c_void_p()
    assert lib.qs_ppo_pop_create(0, d, K, C.byref(h)) == 0
    arr = (QsPpoHyper * K)(*[s.hp for s in solo])
    assert lib.qs_ppo_pop_set_hyper(h, arr, None) == 0
    stats = torch.zeros((K, len(STAT_KEYS)), device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    for it in range(3):
        idx = torch.stack([torch.randperm(R, device=dev, generator=g)[:B] for _ in range(K)])     # [K, B], each agent its own rows
        for a in range(K):
            solo[a].update(obs, act, oldlp, adv, ret, idx[a].contiguous())
        assert lib.qs_ppo_pop_update(h, p(params), p(obs), p(act), p(oldlp), p(adv), p(ret), p(idx), B, B, p(stats), None) == 0
    m, v, st = C.c_void_p(), C.c_void_p(), C.c_void_p()
    assert lib.qs_ppo_pop_state(h, C.byref(m), C.byref(v), C.byref(st)) == 0
    torch.cuda.synchronize()
    npar = params.shape[1]
    pm, pv, ps = _view(m.value, (K, npar), "<f4"), _view(v.value, (K, npar), "<f4"), _view(st.value, (K,), "<i8")
    for a in range(K):
        sm, sv, sst = solo[a].adam_state()
        assert torch.equal(params[a], solo[a].params), a
        assert torch.equal(pm[a], sm) and torch.equal(pv[a], sv) and int(ps[a]) == int(sst[0]) == 3, a
        assert torch.equal(stats[a], solo[a].stats), (a, stats[a], solo[a].stats)
    lib.qs_ppo_pop_destroy(h)
    for s in solo:
        s.close()


def _view(ptr, shape, typestr):
    """A torch view of device memory owned by a library handle."""
    class View:
        pass
    v = View()
    v.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
    return torch.as_tensor(v, device="cuda")


@pytest.mark.parametrize("d", [17, 20])
@pytest.mark.parametrize("noise", [True, False])
@pytest.mark.parametrize("K,n", [(5, 100), (4, 8), (2, 64), (3, 1000)])
def test_population_forward_equals_solo_forward(d, noise, K, n):
    import ctypes as C
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel, unpack_params
    from rl_aerial_manipulator_b200.population import PopulationPPO
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(d * 10 + K)
    blobs = [_perturbed_blob(d, 3 + a) for a in range(K)]
    obs = torch.randn((K * n, d), device=dev, generator=g) * 2
    eps = torch.randn((K * n, 4), device=dev, generator=g) if noise else None
    pop = PopulationPPO.__new__(PopulationPPO)          # the forward wrapper alone, on hand-set attributes
    from rl_aerial_manipulator_b200._cabi import load_library
    from rl_aerial_manipulator_b200.policy import ACTION_HIGH, ACTION_LOW
    pop.lib, pop.K, pop.n, pop.obs_dim, pop.device = load_library(), K, n, d, dev
    pop.params = torch.from_numpy(np.stack(blobs)).to(dev)
    pop._lo, pop._hi = (C.c_float * 4)(*ACTION_LOW), (C.c_float * 4)(*ACTION_HIGH)
    f = lambda *s: torch.full(s, float("nan"), device=dev)   # noqa: E731
    out = pop._forward(obs, eps, (f(K * n, 4), f(K * n, 4), f(K * n), f(K * n)))
    for a in range(K):
        sl = slice(a * n, (a + 1) * n)
        pol = MlpPolicyKernel(unpack_params(blobs[a], d), d, dev, impl="fp32")
        acts, vals, lps = pol.forward(obs[sl].contiguous(), eps[sl].contiguous() if noise else None)
        assert torch.equal(out[0][sl], acts) and torch.equal(out[1][sl], pol.actions_clipped), a
        assert torch.equal(out[2][sl], vals) and torch.equal(out[3][sl], lps), a


def test_row_slice_normal_draws_what_a_solo_buffer_draws():
    dev = torch.device("cuda", 0)
    K, n = 4, 8
    buf = torch.empty((K * n, 4), device=dev)
    gens = [torch.Generator(device=dev).manual_seed(s) for s in SEEDS]
    solo_gens = [torch.Generator(device=dev).manual_seed(s) for s in SEEDS]
    for _ in range(3):
        for a in range(K):
            buf[a * n:(a + 1) * n].normal_(generator=gens[a])
            assert torch.equal(buf[a * n:(a + 1) * n], torch.empty((n, 4), device=dev).normal_(generator=solo_gens[a]))


def _bitwise_equal(x, y):
    """torch.equal on the bit patterns: NaN fields (e.g. last_distance before a first step) compare equal to themselves."""
    ints = {torch.float64: torch.int64, torch.float32: torch.int32}
    if x.dtype in ints:
        return x.dtype == y.dtype and torch.equal(x.contiguous().view(ints[x.dtype]), y.contiguous().view(ints[y.dtype]))
    return torch.equal(x, y)


def _run_pair(env_kw, graph, n_steps=256, batch_size=128, n_epochs=3, state_dict=None, iters=2):
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.population import PopulationPPO
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    K, n = 4, 8
    shared = dict(n_steps=n_steps, batch_size=batch_size, n_epochs=n_epochs, gamma=0.995, gae_lambda=0.9, rollout_graph=graph)
    pop = PopulationPPO(BatchedQuadEnv(K * n, **env_kw), K, SEEDS, hyper=HYPER, state_dicts=None if state_dict is None else [state_dict] * K,
                        **shared)
    plog = []
    pop.learn(iters * n_steps * n, log=plog.append)
    for a in range(K):
        solo = QuadPPO(BatchedQuadEnv(n, env_id_offset=a * n, **env_kw), policy_impl="fp32", seed=SEEDS[a], state_dict=state_dict,
                       **{k: v[a] for k, v in HYPER.items()}, **shared)
        slog = []
        solo.learn(iters * n_steps * n, log=slog.append)
        sl = slice(a * n, (a + 1) * n)
        assert torch.equal(pop.params[a], solo.policy.params), a
        for x, y in zip(pop.adam_state(), solo.opt.adam_state()):
            assert torch.equal(x[a], y.reshape(x[a].shape)), a
        for name in ("obs", "actions", "values", "logp", "rewards", "advantages", "returns", "episode_starts"):
            assert torch.equal(getattr(pop, name)[:, sl], getattr(solo, name)), (a, name)
        ps, ss = pop.env.get_state(), solo.env.get_state()
        for k in ss:
            assert _bitwise_equal(ps[k][sl], ss[k]), (a, k)
        assert torch.equal(pop.env.obs[sl], solo.env.obs) and torch.equal(pop._last_dones[sl], solo._last_dones), a
        mine = [r for r in plog if r["agent"] == a]
        assert len(mine) == len(slog) == iters
        for r, s in zip(mine, slog):
            for k in ("loss", "policy_gradient_loss", "value_loss", "entropy_loss", "grad_norm", "clip_fraction", "approx_kl",
                      "batch_size", "timesteps", "episodes"):
                assert r[k] == s[k], (a, k, r[k], s[k])
            if np.isnan(s["ep_rew_mean"]):
                assert np.isnan(r["ep_rew_mean"])
            else:
                assert abs(r["ep_rew_mean"] - s["ep_rew_mean"]) <= 1e-12 * abs(s["ep_rew_mean"]), (a, r["ep_rew_mean"], s["ep_rew_mean"])
        solo.env.close()
        solo.opt.close()
    episodes = sum(r["episodes"] for r in plog)
    pop.close()
    pop.env.close()
    return episodes


@pytest.mark.parametrize("version", [1, 2])
@pytest.mark.parametrize("graph", [True, False])
def test_population_trains_like_solo_runs(version, graph):
    _run_pair(dict(env_version=version, seed=3), graph)


def test_population_ragged_last_minibatch():
    _run_pair(dict(env_version=1, seed=5), True, batch_size=100)       # 2,048 rows per agent: 20 minibatches of 100 + one of 48


def test_population_dynamics_randomised():
    _run_pair(dict(env_version=2, seed=6, dynamics_randomization=dict(mass=0.2, inertia=0.2, thrust=0.1, wind=0.3)), True)


def test_population_from_shipped_checkpoint(golden_dir):
    z = np.load(os.path.join(golden_dir, "policy_v2.npz"))
    sd = {k[2:]: z[k] for k in z.files if k.startswith("w.")}
    _run_pair(dict(env_version=2, seed=8), True, state_dict=sd)


def test_save_agent_loads_into_quadppo(tmp_path):
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.population import PopulationPPO
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    K, n = 4, 8
    pop = PopulationPPO(BatchedQuadEnv(K * n, env_version=1, seed=2), K, SEEDS, hyper=HYPER, n_steps=64, batch_size=128, n_epochs=2)
    pop.learn(64 * n)
    for a in (0, 2):
        path = str(tmp_path / f"agent{a}.zip")
        pop.save_agent(a, path)
        ppo = QuadPPO.load(path, BatchedQuadEnv(n, env_version=1, env_id_offset=a * n, seed=2), policy_impl="fp32")
        assert torch.equal(ppo.policy.params, pop.params[a])
        m, v, st = ppo.opt.adam_state()
        pm, pv, pst = pop.adam_state()
        assert torch.equal(m, pm[a]) and torch.equal(v, pv[a]) and int(st[0]) == int(pst[a]) == 2 * 4
        assert ppo.num_timesteps == pop.num_timesteps == 64 * n
        assert ppo.ent_coef == HYPER["ent_coef"][a] and ppo.normalize_advantage == HYPER["normalize_advantage"][a]
        ppo.learn(2 * 64 * n)                                        # continues SB3-style from the zip
        assert ppo.num_timesteps == 2 * 64 * n and torch.isfinite(ppo.policy.params).all()
