"""On-device evaluate_policy and EvalCallback on the B200: qs_eval_record against the NumPy restatement of SB3's loop on synthetic
streams (shards, guard rows, graph replay), first-episode evaluation of the shipped v2 policy against the hand loop of the
closed-loop statistics test, auto-reset evaluation against an eager hand loop with SB3's rule (and two shards), stochastic,
VecNormalize and dynamics-randomised evaluation, the early stop, and QuadPPO.learn with an EvalCallback."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from eval_oracle import random_streams, sb3_episodes

pytestmark = pytest.mark.gpu

GUARD = 64


def _env(n, version=2, **kw):
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    return BatchedQuadEnv(n, env_version=version, precision=kw.pop("precision", "f32"), **kw)


def _policy(golden_dir, name="policy_v2.npz"):
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    return MlpPolicyKernel.from_npz(os.path.join(golden_dir, name), device="cuda", impl="tensor")


class _Recorder:
    """qs_eval_begin / qs_eval_record of one shard over synthetic per-step inputs; output buffers carry GUARD sentinel rows."""

    def __init__(self, E, G, off, n, f64):
        from rl_aerial_manipulator_b200 import _cabi, evaluation
        self.lib, dev = _cabi.load_library(), "cuda"
        first, last = evaluation.first_slot(E, G, [off, off + n])
        self.m = int(last - first)
        self.count = torch.zeros(n, dtype=torch.int32, device=dev)
        self.state = torch.zeros(_cabi.EVAL_STATE_WORDS, dtype=torch.int32, device=dev)
        self.out = {"ret": torch.full((self.m + GUARD,), 7.5, dtype=torch.float64, device=dev),
                    "len": torch.full((self.m + GUARD,), -7, dtype=torch.int32, device=dev),
                    "flags": torch.full((self.m + GUARD,), 0xEE, dtype=torch.uint8, device=dev),
                    "step": torch.full((self.m + GUARD,), -9, dtype=torch.int32, device=dev)}
        a = self.a = _cabi.QsEvalArgs()
        a.n, a.env_id_offset, a.n_global, a.n_eval_episodes, a.return_is_f64 = n, off, G, E, int(f64)
        a.count, a.state = self.count.data_ptr(), self.state.data_ptr()
        a.ret_out, a.len_out, a.flags_out, a.step_out = (self.out[k].data_ptr() for k in ("ret", "len", "flags", "step"))
        self.off, self.n = off, n

    def _st(self):
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def begin(self):
        assert self.lib.qs_eval_begin(C.byref(self.a), self._st()) == 0

    def record(self, flags, ret, ln):
        """flags / ret / ln: device rows of the whole batch for one step; this shard reads its slice."""
        sl = slice(self.off, self.off + self.n)
        self.a.flags, self.a.ep_return, self.a.ep_len = flags[sl].data_ptr(), ret[sl].data_ptr(), ln[sl].data_ptr()
        assert self.lib.qs_eval_record(C.byref(self.a), self._st()) == 0, self.lib.qs_eval_last_error()

    def slots(self):
        guards_ok = all(bool((v[self.m:] == v[-1]).all()) and float(v[-1]) == {"ret": 7.5, "len": -7, "flags": 0xEE, "step": -9}[k]
                        for k, v in self.out.items())
        assert guards_ok, "a guard row after an output buffer was written"
        return {k: v[:self.m].cpu().numpy() for k, v in self.out.items()}


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("n", [1, 31, 33, 4097])
def test_record_kernel_equals_sb3_restatement(n, f64):
    rng = np.random.default_rng(n * 2 + int(f64))
    T = 160
    for E in sorted({1, n, 3 * n + 5, max(1, n // 2) + 1}):
        flags, ret, ln = random_streams(rng, T, n, 0.08, f64)
        want = sb3_episodes(E, flags, ret, ln)
        dflags, dret, dln = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (flags, ret, ln))
        shards = [(0, n)] + ([(0, n // 2), (n // 2, n - n // 2)] if n > 1 else [])
        rem_single = None
        for shard_set in ([shards[0]], shards[1:]) if n > 1 else ([shards[0]],):
            recs = [_Recorder(E, n, off, m, f64) for off, m in shard_set]
            rem = np.zeros(T, dtype=np.int64)
            for r in recs:
                r.begin()
            for t in range(T):
                for r in recs:
                    r.record(dflags[t], dret[t], dln[t])
                rem[t] = sum(int(r.state[1]) for r in recs)
            np.testing.assert_array_equal(rem, want["remaining"], err_msg=f"n={n} E={E} shards={shard_set}")
            assert all(int(r.state[0]) == T for r in recs)
            got = {k: np.concatenate([r.slots()[k] for r in recs]) for k in ("ret", "len", "flags", "step")}
            filled = np.zeros(E, dtype=bool)
            tgt_counts = np.concatenate([r.count.cpu().numpy() for r in recs])
            for i in range(n):
                filled[want["base"][i]:want["base"][i] + tgt_counts[i]] = True
            for k in got:
                np.testing.assert_array_equal(got[k][filled], want["slot_" + k][filled], err_msg=f"{k} n={n} E={E}")
            if rem_single is None:
                rem_single = got
            else:
                for k in got:
                    np.testing.assert_array_equal(got[k], rem_single[k])
        # graph replay of the same T steps: bit-identical to eager
        rec = _Recorder(E, n, 0, n, f64)
        rec.begin()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for t in range(T):
                rec.record(dflags[t], dret[t], dln[t])
        rec.begin()
        g.replay()
        torch.cuda.synchronize()
        got = rec.slots()
        for k in got:
            np.testing.assert_array_equal(got[k], rem_single[k])
        assert int(rec.state[0]) == T and int(rec.state[1]) == want["remaining"][-1]


def _hand_loop(policy, env, E, T_max, deterministic=True, seed=0, stats=None, poll=64):
    """The eager loop evaluate_policy replaces: forward -> step on the clipped actions, per-step outputs brought to the host, SB3's
    rule applied afterwards by the NumPy restatement."""
    obs = env.reset()
    if not deterministic:
        if getattr(policy, "_philox_counter", None) is None:
            policy._philox_counter = torch.zeros(2, dtype=torch.int64, device=env.device)
        policy._philox_counter.zero_()
    fl, rt, ln = [], [], []
    off = int(env.cfg.env_id_offset)
    for t in range(T_max):
        if deterministic:
            policy.forward(obs, None, norm_stats=stats)
        else:
            policy.forward_sampled(obs, seed, off, norm_stats=stats)
        out = env.step(policy.actions_clipped)
        obs = out.obs
        fl.append(out.flags.cpu().numpy().copy())
        rt.append(out.ep_return.double().cpu().numpy().copy())
        ln.append(out.ep_len.cpu().numpy().copy())
        if t % poll == poll - 1:            # done when every env has finished as many episodes as its target
            dones = ((np.stack(fl) & 3) != 0).sum(0)
            if not (dones < (E + np.arange(env.n_envs)) // env.n_envs).any():
                break
    want = sb3_episodes(E, np.stack(fl), np.stack(rt), np.stack(ln))
    assert want["remaining"][-1] == 0
    return want


def _assert_same(res, want):
    np.testing.assert_array_equal(res.ep_return.cpu().numpy(), want["ret"])
    np.testing.assert_array_equal(res.ep_length.cpu().numpy(), want["len"])
    np.testing.assert_array_equal(res.flags.cpu().numpy(), want["flags"])
    np.testing.assert_array_equal(res.step.cpu().numpy(), want["step"])
    np.testing.assert_array_equal(res.env_id.cpu().numpy(), want["env_id"])


def test_first_episode_evaluation_of_shipped_v2_policy(golden_dir):
    """E = n = 4,096 on an auto_reset=False batch with the golden seed: one episode per env, the loop of
    test_closed_loop_statistics_vs_reference (same kernels, so the same episodes bit for bit) and its statistics windows."""
    from rl_aerial_manipulator_b200.evaluation import evaluate, evaluate_policy
    g = np.load(os.path.join(golden_dir, "closed_loop_v2.npz"))
    n = 4096
    pol = _policy(golden_dir)
    mk = lambda: _env(n, auto_reset=False, seed=int(g["seed"]))   # a fresh handle per run: every reset starts the next episode
    res = evaluate(pol, mk(), n)
    # the hand loop of the closed-loop statistics test, plus the Monitor return the env reports at the first done
    env = mk()
    obs = env.reset()
    length = torch.zeros(n, dtype=torch.int32, device="cuda")
    ret = torch.zeros(n, dtype=torch.float64, device="cuda")
    mon = torch.zeros(n, dtype=torch.float64, device="cuda")
    fin_flags = torch.zeros(n, dtype=torch.uint8, device="cuda")
    done = torch.zeros(n, dtype=torch.bool, device="cuda")
    for t in range(2100):
        pol.forward(obs, None)
        out = env.step(pol.actions_clipped)
        obs = out.obs
        ret += torch.where(done, 0.0, out.reward.double())
        newly = out.done & ~done
        length[newly] = t + 1
        fin_flags[newly] = out.flags[newly]
        mon[newly] = out.ep_return[newly].double()
        done |= newly
        if t % 64 == 63 and bool(done.all()):
            break
    assert bool(done.all())
    by_env = torch.argsort(res.env_id)
    np.testing.assert_array_equal(res.ep_length[by_env].cpu().numpy(), length.cpu().numpy())
    np.testing.assert_array_equal(res.flags[by_env].cpu().numpy(), fin_flags.cpu().numpy())
    np.testing.assert_array_equal(res.ep_return[by_env].cpu().numpy(), mon.cpu().numpy())
    np.testing.assert_array_equal(res.step[by_env].cpu().numpy() + 1, length.cpu().numpy())
    # Monitor's return is the env's float32 running sum; the hand loop sums the float32 rewards in float64
    np.testing.assert_allclose(res.ep_return[by_env].cpu().numpy(), ret.cpu().numpy(), rtol=1e-4)
    lengths, flags, rets = res.ep_length.cpu().numpy().astype(np.float64), res.flags.cpu().numpy(), res.ep_return.cpu().numpy()
    success = ((flags & 0x04) != 0) & ((flags & 0x01) != 0)
    assert res.success_rate == success.mean() >= 0.94
    se_len, se_ret = g["length"].std() / np.sqrt(64), g["ep_return"].std() / np.sqrt(64)
    assert abs(lengths[success].mean() - g["length"].mean()) <= 3.5 * se_len
    assert abs(rets[success].mean() - g["ep_return"].mean()) <= 3.5 * se_ret
    assert res.mean_length_successful == pytest.approx(lengths[success].mean())
    assert res.crash_rate + res.oob_rate + res.truncation_rate <= 1 - res.success_rate + 1e-12
    assert res.steps <= int(lengths.max()) + 64                         # the early stop
    mean, std = evaluate_policy(pol, mk(), n)
    r6 = [round(float(x), 6) for x in rets]
    assert mean == float(np.mean(r6)) and std == float(np.std(r6))
    with pytest.raises(ValueError, match="auto-reset"):
        evaluate_policy(pol, env, n + 1)
    env.close()


def test_auto_reset_evaluation_equals_hand_loop_and_shards(golden_dir):
    from rl_aerial_manipulator_b200.evaluation import EvalResult, evaluate, evaluate_policy
    n = 256
    E = 3 * n + 5
    pol = _policy(golden_dir)
    mk = lambda: _env(n, seed=3)
    res = evaluate(pol, mk(), E, poll_every=32)
    want = _hand_loop(pol, mk(), E, 9000)
    _assert_same(res, want)
    assert res.steps <= int(res.step.max()) + 1 + 32
    env = mk()
    rewards, lengths = evaluate_policy(pol, env, E, return_episode_rewards=True)
    assert rewards == [round(float(x), 6) for x in want["ret"]] and lengths == want["len"].tolist()
    with pytest.raises(AssertionError, match="threshold"):
        evaluate_policy(pol, env, E, reward_threshold=1e12)
    with pytest.raises(ValueError, match="render"):
        evaluate_policy(pol, env, E, render=True)
    with pytest.raises(ValueError, match="callback"):
        evaluate_policy(pol, env, E, callback=lambda *_: None)
    # two half-shards (same seed, env_id_offset): together exactly the single handle's records
    parts = []
    for off in (0, n // 2):
        shard = _env(n // 2, seed=3, env_id_offset=off)
        parts.append(evaluate(pol, shard, E, n_global=n, poll_every=32))
        shard.close()
    _assert_same(EvalResult.concat(parts), want)
    env.close()


def test_stochastic_evaluation(golden_dir):
    from rl_aerial_manipulator_b200.evaluation import evaluate
    n, E = 128, 200
    pol = _policy(golden_dir)
    mk = lambda: _env(n, seed=5)
    a = evaluate(pol, mk(), E, deterministic=False, noise_seed=11)
    b = evaluate(pol, mk(), E, deterministic=False, noise_seed=11)
    c = evaluate(pol, mk(), E, deterministic=False, noise_seed=12)
    for f in ("ep_return", "ep_length", "flags", "step", "env_id"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    assert not torch.equal(a.ep_return, c.ep_return)
    _assert_same(a, _hand_loop(pol, mk(), E, 9000, deterministic=False, seed=11))     # graph replays == eager steps


def test_vecnormalize_evaluation_equals_hand_loop(golden_dir):
    """Plumbing parity: a v1 env, the 17-D golden VecNormalize statistics and the v1 golden policy (not a claim that this pairing
    flies well); the statistics are read only."""
    from rl_aerial_manipulator_b200.evaluation import evaluate
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    n, E = 256, 300
    pol = _policy(golden_dir, "policy_v1.npz")
    mk = lambda: _env(n, version=1, seed=7)
    env = mk()
    vn = DeviceVecNormalize(env, training=False)
    z = np.load(os.path.join(golden_dir, "vecnorm_v1.npz"))
    vn.load_state_dict({k: z[k] for k in z.files})
    before = vn.obs_rms.stats.clone()
    res = evaluate(pol, env, E, vecnorm=vn)
    assert torch.equal(vn.obs_rms.stats, before)
    _assert_same(res, _hand_loop(pol, mk(), E, 6000, stats=vn.obs_rms.stats))
    assert torch.equal(vn.obs_rms.stats, before)


def test_dynamics_randomised_env_evaluates(golden_dir):
    from rl_aerial_manipulator_b200.evaluation import evaluate
    n, E = 512, 1000
    env = _env(n, seed=9, dynamics_randomization=dict(mass=0.2, inertia=0.2, thrust=0.1, wind=0.3))
    res = evaluate(_policy(golden_dir), env, E)
    assert res.ep_return.numel() == E and 0.0 < res.success_rate <= 1.0
    assert res.steps <= int(res.step.max()) + 1 + 64
    env.close()


def test_quadppo_eval_callback(golden_dir):
    from rl_aerial_manipulator_b200.evaluation import EvalCallback
    from rl_aerial_manipulator_b200.policy import unpack_params
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    n, T = 512, 32

    def run(with_cb):
        env = _env(n, seed=1)
        vn = DeviceVecNormalize(env)
        ppo = QuadPPO(env, vecnorm=vn, n_steps=T, batch_size=4096, n_epochs=2, policy_impl="fp32", seed=0, rollout_graph=True)
        logs, snaps = [], []
        cb = EvalCallback(_env(64, seed=2), eval_freq=T, n_eval_episodes=96) if with_cb else None

        def log(d):
            logs.append(d)
            snaps.append((ppo.policy.params.clone(), vn.obs_rms.stats.clone()))
        ppo.learn(3 * T * n, log=log, callback=cb)
        if with_cb:
            with pytest.raises(ValueError, match="training env"):
                ppo.learn(4 * T * n, callback=EvalCallback(env, eval_freq=T))
        return ppo, logs, snaps, cb

    ppo0, logs0, _, _ = run(False)
    ppo1, logs1, snaps, cb = run(True)
    assert torch.equal(ppo0.policy.params, ppo1.policy.params)           # evaluation does not change training
    assert len(logs1) == 3 and all("eval/mean_reward" in l and "eval/success_rate" in l for l in logs1)
    assert not any(k.startswith("eval/") for l in logs0 for k in l)
    best = int(np.argmax([l["eval/mean_reward"] for l in logs1]))
    assert cb.best_mean_reward == logs1[best]["eval/mean_reward"]
    sd = cb.best_state_dict()
    want = unpack_params(snaps[best][0].cpu().numpy(), ppo1.env.obs_dim)
    assert sd["policy"].keys() == want.keys() and all(np.array_equal(sd["policy"][k], want[k]) for k in want)
    d = ppo1.env.obs_dim
    np.testing.assert_array_equal(sd["vecnorm"]["obs_mean"], snaps[best][1][1:1 + d].cpu().numpy())
    np.testing.assert_array_equal(sd["vecnorm"]["obs_var"], snaps[best][1][1 + d:].cpu().numpy())
