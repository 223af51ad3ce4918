"""QuadPPO.save / load and the checkpoint callbacks on the device: exact resume bit for bit, SB3-semantics resume against torch's
Adam, the refusals, and callbacks that leave training unchanged."""
import os

import numpy as np
import pytest
import torch

from test_ppo import random_minibatch

pytestmark = pytest.mark.gpu

RUN = dict(n_envs=512, n_steps=16, batch_size=2048, n_epochs=2, policy_impl="fp32", rollout_graph=True, version=2, vecnorm=True,
           norm_reward=False, dyn=None)
CASES = {
    "v1_vecnorm_norm_reward": dict(version=1, norm_reward=True),
    "v2_no_vecnorm": dict(vecnorm=False),
    "eager_collection": dict(rollout_graph=False),
    "dynamics_randomised": dict(dyn=dict(mass=0.2, inertia=0.2, thrust=0.1, wind=0.3)),
    "compacted_bootstrap_131072_envs": dict(n_envs=131072, n_steps=8, batch_size=65536, n_epochs=1, policy_impl="auto"),
}


def _env_vn(c, seed=1, dyn="same"):
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    env = BatchedQuadEnv(c["n_envs"], env_version=c["version"], precision="f32", seed=seed,
                         dynamics_randomization=c["dyn"] if dyn == "same" else dyn)
    vn = DeviceVecNormalize(env, norm_reward=c["norm_reward"], gamma=0.995) if c["vecnorm"] else None
    return env, vn


def _ppo(c, env, vn):
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    return QuadPPO(env, vecnorm=vn, n_steps=c["n_steps"], batch_size=c["batch_size"], n_epochs=c["n_epochs"], seed=0,
                   policy_impl=c["policy_impl"], rollout_graph=c["rollout_graph"])


def _load(c, path, env, vn, **kw):
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    return QuadPPO.load(path, env, vn, policy_impl=c["policy_impl"], rollout_graph=c["rollout_graph"], **kw)


def _snapshot(ppo, logs):
    """Everything the comparison covers, as host bytes: parameters, Adam m/v/step, VecNormalize statistics, the last rollout's
    buffers, the env state, and the logged ep_rew_mean."""
    m, v, st = ppo.opt.adam_state()
    t = {"params": ppo.policy.params, "adam_m": m, "adam_v": v, "adam_step": st}
    for k in ("obs", "actions", "values", "logp", "rewards", "advantages", "returns", "episode_starts"):
        t[k] = getattr(ppo, k)
    if ppo.vecnorm is not None:
        t["obs_rms"], t["ret_rms"], t["vn_returns"] = ppo.vecnorm.obs_rms.stats, ppo.vecnorm.ret_rms.stats, ppo.vecnorm.returns
    t.update({f"env.{k}": x for k, x in ppo.env.get_state().items()})
    out = {k: x.detach().cpu().numpy().tobytes() for k, x in t.items()}
    out["ep_rew_mean"] = np.float64(logs[-1]["ep_rew_mean"]).tobytes()
    out["timesteps"] = logs[-1]["timesteps"]
    return out


def _assert_same(a, b):
    assert a.keys() == b.keys()
    diff = [k for k in a if a[k] != b[k]]
    assert not diff, f"differ bitwise: {diff}"


def _uninterrupted(c, iters=4):
    env, vn = _env_vn(c)
    ppo, logs = _ppo(c, env, vn), []
    ppo.learn(iters * c["n_steps"] * c["n_envs"], log=logs.append)
    return _snapshot(ppo, logs)


@pytest.mark.parametrize("case", list(CASES))
def test_exact_resume_is_bitwise(case, tmp_path):
    """Train 2 iterations, save, load into a fresh env / VecNormalize / QuadPPO, train to 4: bitwise the 4 uninterrupted ones."""
    c = dict(RUN, **CASES[case])
    want = _uninterrupted(c)
    per = c["n_steps"] * c["n_envs"]
    env, vn = _env_vn(c)
    ppo = _ppo(c, env, vn)
    ppo.learn(2 * per)
    path = str(tmp_path / "ckpt.zip")
    ppo.save(path)
    env2, vn2 = _env_vn(c)
    ppo2 = _load(c, path, env2, vn2)
    assert ppo2.num_timesteps == 2 * per and ppo2._n_updates == 2 * c["n_epochs"]
    logs = []
    ppo2.learn(4 * per, log=logs.append)
    assert len(logs) == 2
    _assert_same(_snapshot(ppo2, logs), want)


def test_save_before_training_then_resume(tmp_path):
    """A checkpoint written before the first collection resumes like a fresh run (the env is reset at the first collection)."""
    c = dict(RUN)
    want = _uninterrupted(c, iters=2)
    env, vn = _env_vn(c)
    path = str(tmp_path / "fresh.zip")
    _ppo(c, env, vn).save(path)
    env2, vn2 = _env_vn(c)
    ppo2, logs = _load(c, path, env2, vn2), []
    ppo2.learn(2 * c["n_steps"] * c["n_envs"], log=logs.append)
    _assert_same(_snapshot(ppo2, logs), want)


def test_sb3_semantics_resume_matches_torch_adam(golden_dir, tmp_path):
    """A zip as SB3 writes it (no resume member): the shipped v2 weights and a torch Adam stepped on the CPU.  After load, one
    minibatch update on a fixed batch matches oracle.ppo_oracle.torch_update continuing from the same Adam state."""
    from oracle import ppo_oracle as po
    from rl_aerial_manipulator_b200 import sb3_compat as sc
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.policy import pack_params
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    z = np.load(os.path.join(golden_dir, "policy_v2.npz"))
    sd = {k[2:]: z[k].astype(np.float32) for k in z.files if k.startswith("w.")}
    D, B, hp = 20, 256, dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5)
    net = po.make_torch_actor_critic(sd, D)
    opt = torch.optim.Adam(net.parameters(), lr=2e-4, eps=1e-5)
    rng = np.random.default_rng(3)
    for _ in range(3):
        po.torch_update(net, opt, tuple(torch.from_numpy(x) for x in random_minibatch(rng, B, D, sd)), **hp)
    data = {"num_timesteps": 49152, "_n_updates": 30, "n_steps": 2048, "batch_size": 128, "n_epochs": 10, "gamma": 0.995,
            "gae_lambda": 0.9, "learning_rate": 2e-4, "normalize_advantage": True, **hp}
    path = str(tmp_path / "sb3.zip")
    sc.save_model_zip(path, {k: v.detach().numpy() for k, v in net.state_dict().items()}, opt.state_dict(), data)
    env = BatchedQuadEnv(64, env_version=2, seed=1)
    ppo = QuadPPO.load(path, env, n_steps=8, policy_impl="fp32")
    assert ppo.num_timesteps == 49152 and ppo.batch_size == 128 and ppo.ent_coef == 0.01 and ppo._last_obs is None
    batch = random_minibatch(rng, B, D, {k: v.detach().numpy() for k, v in net.state_dict().items()})
    ppo.opt.update(*(torch.from_numpy(x).cuda() for x in batch))
    po.torch_update(net, opt, tuple(torch.from_numpy(x) for x in batch), **hp)
    blob = lambda f: pack_params({n: f(p) for n, p in net.named_parameters()}, D)
    m, v, st = (x.cpu().numpy() for x in ppo.opt.adam_state())
    np.testing.assert_allclose(ppo.policy.params.cpu().numpy(), blob(lambda p: p.detach().numpy()), rtol=0, atol=1e-5)
    np.testing.assert_allclose(m, blob(lambda p: opt.state[p]["exp_avg"].numpy()), rtol=0, atol=1e-5)
    np.testing.assert_allclose(v, blob(lambda p: opt.state[p]["exp_avg_sq"].numpy()), rtol=0, atol=1e-5)
    assert int(st[0]) == 4


def test_refusals_and_sb3_path_on_mismatch(tmp_path):
    c = dict(RUN, dyn=dict(mass=0.2))
    env, vn = _env_vn(c)
    ppo = _ppo(c, env, vn)
    ppo.learn(c["n_steps"] * c["n_envs"])
    path = str(tmp_path / "ckpt.zip")
    with pytest.raises(ValueError, match="single-rank"):
        ppo.world = 2
        ppo.save(path)
    ppo.world = 1
    ppo.save(path)
    for kw, field in ((dict(seed=2), "seed"), (dict(dyn=None), "dynamics_randomization")):
        env2, vn2 = _env_vn(c, **kw)
        with pytest.raises(ValueError, match=field):
            _load(c, path, env2, vn2)
    with pytest.raises(ValueError, match="vecnorm"):
        _load(c, path, _env_vn(c)[0], None)
    env3, vn3 = _env_vn(c, seed=2)
    ppo3 = _load(c, path, env3, vn3, resume_env_state=False)           # SB3 semantics: weights + Adam, env reset at first collection
    assert ppo3._last_obs is None and ppo3.num_timesteps == ppo.num_timesteps
    assert torch.equal(ppo3.policy.params, ppo.policy.params)
    assert all(torch.equal(a, b) for a, b in zip(ppo3.opt.adam_state(), ppo.opt.adam_state()))
    ppo3.learn(2 * c["n_steps"] * c["n_envs"])
    assert ppo3.num_timesteps == 2 * c["n_steps"] * c["n_envs"]


def test_callbacks_write_resumable_checkpoints_and_leave_training_unchanged(tmp_path):
    from rl_aerial_manipulator_b200 import sb3_compat as sc
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.evaluation import CheckpointCallback, EvalCallback
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    c = dict(RUN)
    T, n = c["n_steps"], c["n_envs"]
    want = _uninterrupted(c)
    env, vn = _env_vn(c)
    ppo, logs = _ppo(c, env, vn), []
    ck = CheckpointCallback(T, str(tmp_path / "ckpt"), save_vecnormalize=True)
    ev = EvalCallback(BatchedQuadEnv(64, env_version=2, seed=2), eval_freq=T, n_eval_episodes=64, best_model_save_path=str(tmp_path / "best"))
    ppo.learn(4 * T * n, log=logs.append, callback=[ck, ev])
    _assert_same(_snapshot(ppo, logs), want)                        # callbacks only read device state
    assert all("eval/mean_reward" in l for l in logs)
    names = sorted(os.listdir(tmp_path / "ckpt"))
    assert names == sorted([f"rl_model_{i * T * n}_steps.zip" for i in range(1, 5)] +
                           [f"rl_model_vecnormalize_{i * T * n}_steps.pkl" for i in range(1, 5)])
    assert sorted(os.listdir(tmp_path / "best")) == ["best_model.zip", "best_model_vecnormalize.pkl"]
    best = ev.best_state_dict()
    pol = MlpPolicyKernel.from_sb3_zip(str(tmp_path / "best" / "best_model.zip"))
    assert all(np.array_equal(pol.state_dict[k], best["policy"][k]) for k in best["policy"])
    bvn = sc.load_vecnormalize_pkl(str(tmp_path / "best" / "best_model_vecnormalize.pkl"))
    assert np.array_equal(bvn["obs_mean"], best["vecnorm"]["obs_mean"]) and np.array_equal(bvn["obs_var"], best["vecnorm"]["obs_var"])
    # the reference's resume flow: load the middle checkpoint and its vec_normalize.pkl, finish the run
    mid = tmp_path / "ckpt" / f"rl_model_{2 * T * n}_steps.zip"
    env2, vn2 = _env_vn(c)
    vn2.load_state_dict(sc.load_vecnormalize_pkl(str(tmp_path / "ckpt" / f"rl_model_vecnormalize_{2 * T * n}_steps.pkl")))
    ppo2, logs2 = _load(c, str(mid), env2, vn2), []
    ppo2.learn(4 * T * n, log=logs2.append)
    _assert_same(_snapshot(ppo2, logs2), want)
