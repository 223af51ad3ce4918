"""Dynamics randomisation on the B200: the per-episode draw (qs_dynamics_randomization / qs_get_dynamics) against the NumPy
restatement, redraws at exactly the resets, zero ranges == the nominal kernels, one randomised step against the oracle's direct
physical form, qs_step_many / qs_step_range / fused moments on an armed handle, PPO on an armed env, and the refusals."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import dyn_oracle as do
from test_dynamics_cpu import _random_batch
from test_gpu_parity import make_env, push_batch, t2n

pytestmark = pytest.mark.gpu

DR = dict(mass=0.3, inertia=0.25, thrust=0.15, wind=0.4, seed=77)
RANGES = (0.3, 0.25, 0.15, 0.4)


def rows(env):
    d = env.dynamics()
    return torch.cat([d["mass_scale"][:, None], d["inertia_scale"][:, None], d["thrust_scale"], d["wind"]], 1).cpu().numpy()


def draw(n, episodes, offset=0):
    return do.dynamics_draw(DR["seed"], *RANGES, np.arange(n) + offset, episodes)


def crash_prone(env, frac=3):
    """A third of the envs just above the crash height and sinking: terminations and auto-resets within a few steps."""
    n = env.n_envs
    y = env.get_state(["y"])["y"]
    y[: n // frac, 2] = 0.13
    y[: n // frac, 5] = -0.5
    env.set_state(y=y)


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("variant", ["v2", "v1", "v2m"])
def test_draw_equals_numpy_restatement(variant, precision):
    n = 3000
    env = make_env(n, variant, precision=precision, dynamics_randomization=DR)
    env.reset()
    want = draw(n, np.zeros(n))
    got = rows(env)
    if precision == "f64":
        np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64))
    else:
        np.testing.assert_array_equal(got, want.astype(np.float32).astype(np.float64))


def test_sharded_handles_draw_the_unsharded_batch():
    n = 2048
    full = make_env(n, "v2", precision="f64", dynamics_randomization=DR)
    full.reset()
    halves = [make_env(n // 2, "v2", precision="f64", env_id_offset=o, dynamics_randomization=DR) for o in (0, n // 2)]
    for h in halves:
        h.reset()
    np.testing.assert_array_equal(np.concatenate([rows(h) for h in halves]), rows(full))


def test_ragged_batch_leaves_guard_rows_untouched():
    n = 1000
    env = make_env(n, "v1", precision="f32", dynamics_randomization=DR)
    env.reset()
    out = torch.full((n + 40, 9), -123.5, dtype=torch.float64, device="cuda")
    rc = env.lib.qs_get_dynamics(env._h, C.c_void_p(out.data_ptr()), env._stream())
    assert rc == 0
    o = t2n(out)
    assert np.all(o[n:] == -123.5)
    np.testing.assert_array_equal(o[:n], draw(n, np.zeros(n)).astype(np.float32).astype(np.float64))


def test_arming_after_reset_draws_the_current_episode():
    n = 512
    env = make_env(n, "v2", precision="f64")
    env.reset()
    env.set_state(episode=np.arange(n, dtype=np.int32) % 7)
    env.randomize_dynamics(DR)
    np.testing.assert_array_equal(rows(env), draw(n, np.arange(n) % 7))


def test_redrawn_exactly_at_resets_qs_step_and_mask():
    n = 4096
    env = make_env(n, "v2", precision="f32", dynamics_randomization=DR)
    env.reset()
    crash_prone(env)
    g = torch.Generator(device="cuda").manual_seed(0)
    n_reset = 0
    for t in range(30):
        before, ep0 = rows(env), t2n(env.get_state(["episode"])["episode"])
        a = torch.rand((n, 4), device="cuda", generator=g) * torch.tensor([2.0, 2, 2, 2], device="cuda") - torch.tensor([0.0, 1, 1, 1], device="cuda")
        out = env.step(a)
        done, after, ep1 = t2n(out.done), rows(env), t2n(env.get_state(["episode"])["episode"])
        np.testing.assert_array_equal(ep1, ep0 + done)
        np.testing.assert_array_equal(after[~done], before[~done])                   # constant within an episode
        np.testing.assert_array_equal(after[done], draw(n, ep1).astype(np.float32).astype(np.float64)[done])
        n_reset += done.sum()
    assert n_reset >= n // 4
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[::3] = 1
    before, ep0 = rows(env), t2n(env.get_state(["episode"])["episode"])
    env.reset(mask)
    m = t2n(mask).astype(bool)
    after, ep1 = rows(env), t2n(env.get_state(["episode"])["episode"])
    np.testing.assert_array_equal(ep1, ep0 + m)
    np.testing.assert_array_equal(after[~m], before[~m])
    np.testing.assert_array_equal(after[m], draw(n, ep1).astype(np.float32).astype(np.float64)[m])


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_step_many_redraws_mid_launch_and_equals_single_steps(precision):
    """qs_step_many keeps the parameters in registers and redraws them at an in-kernel auto-reset: T = 24 steps in one launch ==
    24 calls of qs_step on a twin handle (tolerances of test_gpu_step_many.py), parameters after the launch == the draw of every
    env's final episode."""
    n, T = 4099, 24
    env_m = make_env(n, "v2", precision=precision, seed=3, dynamics_randomization=DR)
    env_s = make_env(n, "v2", precision=precision, seed=3, dynamics_randomization=DR)
    for e in (env_m, env_s):
        e.reset()
        crash_prone(e)
    g = torch.Generator(device="cuda").manual_seed(5)
    acts = (torch.tensor([0.0, -1, -1, -1], device="cuda") + 2.0 * torch.rand((T, n, 4), device="cuda", generator=g)).contiguous()
    out = env_m.step_many(T, actions=acts)
    fl_m, rew_m, obs_m = out["flags"].clone(), out["reward"].clone(), out["obs"].clone()
    done_any = t2n(((fl_m & 3) != 0).any(0))
    assert done_any.sum() >= n // 10
    ep = t2n(env_m.get_state(["episode"])["episode"])
    want = draw(n, ep)
    if precision == "f32":
        want = want.astype(np.float32).astype(np.float64)
    np.testing.assert_array_equal(rows(env_m), want)
    tol = dict(rtol=1e-5, atol=1e-5) if precision == "f32" else dict(rtol=1e-12, atol=1e-12)
    for t in range(T):
        s = env_s.step(acts[t])
        same = s.flags == fl_m[t]
        assert int((~same).sum()) <= max(1, n // 2000), f"t={t}"
        if not bool(same.all()):                 # an ulp across a threshold: the twins diverge from here on
            return
        torch.testing.assert_close(s.obs, obs_m[t], **tol)
        torch.testing.assert_close(s.reward, rew_m[t], rtol=1e-4 if precision == "f32" else 1e-11, atol=2e-3 if precision == "f32" else 1e-9)
    np.testing.assert_array_equal(rows(env_s), rows(env_m))


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_zero_ranges_reproduce_the_nominal_kernel(precision):
    """All ranges 0: k_m = k_I = eta = 1 and no wind, so the randomised kernel computes the nominal physics.  Multiplying by 1
    and adding 0 are exact, but the two kernels are different code, so nvcc may contract a*b+c into FMAs at other places:
    obs / reward agree to 1e-6 (float32) / 1e-13 (float64) rather than bit for bit; flags are equal."""
    n = 8192
    zero = dict(mass=0.0, inertia=0.0, thrust=0.0, wind=0.0)
    env_d = make_env(n, "v2", precision=precision, seed=9, dynamics_randomization=zero)
    env_n = make_env(n, "v2", precision=precision, seed=9)
    env_d.reset(), env_n.reset()
    assert np.all(rows(env_d) == [1, 1, 1, 1, 1, 1, 0, 0, 0])
    g = torch.Generator(device="cuda").manual_seed(1)
    tol = 1e-6 if precision == "f32" else 1e-13
    n_done = 0
    for t in range(200):
        a = (torch.tensor([0.0, -1, -1, -1], device="cuda") + 2.0 * torch.rand((n, 4), device="cuda", generator=g)).contiguous()
        od, on = env_d.step(a), env_n.step(a)
        assert torch.equal(od.flags, on.flags), t
        torch.testing.assert_close(od.obs, on.obs, rtol=tol, atol=tol)
        torch.testing.assert_close(od.reward, on.reward, rtol=tol, atol=tol * 100)
        n_done += int(od.done.sum())
        env_d.set_state(**env_n.get_state())                        # no drift: every step compares one step from the same state
    assert n_done > 0


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("variant", ["v2", "v1", "v2m"])
def test_one_step_vs_dyn_oracle(variant, precision):
    """set_state + set_dynamics with random parameters, one step, against the oracle's direct physical form: float64 RK4 1e-12
    relative, float32 1e-4; flags exact away from thresholds."""
    n = 8192
    rng = np.random.default_rng({"v2": 1, "v1": 2, "v2m": 3}[variant])
    b = _random_batch(rng, variant, n)
    dyn = do.dynamics_draw(123, 0.4, 0.4, 0.3, 0.6, np.arange(n), np.zeros(n))
    dyn[: n // 20, 2] = 0.0
    if precision == "f32":
        dyn = dyn.astype(np.float32).astype(np.float64)
    a = np.stack([rng.uniform(0, 2, n), *rng.uniform(-1, 1, (3, n))], 1).astype(np.float32)
    env = make_env(n, variant, precision=precision, auto_reset=False, dynamics_randomization=DR)
    push_batch(env, b)
    env.set_dynamics(mass_scale=dyn[:, 0], inertia_scale=dyn[:, 1], thrust_scale=dyn[:, 2:6], wind=dyn[:, 6:9])
    np.testing.assert_array_equal(rows(env), dyn)
    out = env.step(torch.from_numpy(a).cuda())
    with np.errstate(all="ignore"):
        obs, rew, term, trunc, info = do.step(b, a, substeps=1, **do.dyn_kwargs(dyn))
    st = {k: t2n(v) for k, v in env.get_state().items()}
    want = term.astype(np.uint8) | (trunc.astype(np.uint8) << 1) | ((info & 0xF) << 2)
    flags = t2n(out.flags)
    if precision == "f64":
        np.testing.assert_allclose(st["y"], b.y, rtol=1e-12, atol=1e-13)
        assert (flags != want).sum() <= 2
        same = flags == want
        np.testing.assert_allclose(t2n(out.reward)[same], rew[same], rtol=1e-10, atol=1e-10)
        np.testing.assert_allclose(t2n(out.obs)[same], obs[same], rtol=2e-7, atol=1e-12)
    else:
        np.testing.assert_allclose(st["y"], b.y, rtol=1e-4, atol=1e-4)
        assert (flags != want).mean() < 1e-3
        same = flags == want
        np.testing.assert_allclose(t2n(out.obs)[same], obs[same], rtol=1e-4, atol=1e-4)
    assert (flags != 0).sum() > n // 10


def test_chunked_step_range_equals_single_launch():
    n = 4096 + 100
    envs = [make_env(n, "v2", precision="f32", seed=4, dynamics_randomization=DR) for _ in range(2)]
    for e in envs:
        e.reset()
        crash_prone(e)
    g = torch.Generator(device="cuda").manual_seed(2)
    for t in range(12):
        a = (torch.tensor([0.0, -1, -1, -1], device="cuda") + 2.0 * torch.rand((n, 4), device="cuda", generator=g)).contiguous()
        o1 = envs[0].step(a)
        for first in range(0, n, 1024):
            cnt = min(1024, n - first)
            envs[1].step_range(first, cnt, a[first:first + cnt].contiguous())
        assert torch.equal(o1.obs, envs[1].obs) and torch.equal(o1.reward, envs[1].reward) and torch.equal(o1.flags, envs[1].flags)
    np.testing.assert_array_equal(rows(envs[0]), rows(envs[1]))


def test_fused_moments_on_armed_handle():
    n = 65536
    env = make_env(n, "v2", precision="f32", dynamics_randomization=DR)
    env.reset()
    mom = torch.zeros(1 + 2 * 20, dtype=torch.float64, device="cuda")
    env.fuse_obs_moments(mom)
    a = (torch.tensor([0.0, -1, -1, -1], device="cuda") + 2.0 * torch.rand((n, 4), device="cuda")).contiguous()
    for _ in range(3):
        out = env.step(a)
    x = out.obs.double()
    assert mom[0].item() == n
    torch.testing.assert_close(mom[1:21], x.mean(0), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(mom[21:] / n, x.var(0, unbiased=False), rtol=1e-6, atol=1e-6)
    env.fuse_obs_moments(None)


def test_ppo_on_armed_env_two_graph_iterations():
    """QuadPPO with VecNormalize and the graph-replayed collection on an armed env: two iterations, finite losses, the parameters
    move, and the envs that finished episodes inside the rollouts fly their new episode's airframe."""
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize
    n, T = 512, 32
    env = make_env(n, "v2", precision="f32", dynamics_randomization=DR)
    env.reset()
    crash_prone(env)
    vn = DeviceVecNormalize(env)
    ppo = QuadPPO(env, vecnorm=vn, n_steps=T, batch_size=4096, n_epochs=2, policy_impl="fp32", seed=0, rollout_graph=True)
    p0 = ppo.policy.params.clone()
    logs = []
    ppo.learn(2 * T * n, log=logs.append)
    assert len(logs) == 2 and all(np.isfinite(v) for l in logs for k, v in l.items() if k.endswith("loss"))
    assert float((ppo.policy.params - p0).abs().max()) > 1e-5 and bool(torch.isfinite(ppo.policy.params).all())
    ep = t2n(env.get_state(["episode"])["episode"])
    assert (ep > 0).sum() >= n // 4
    np.testing.assert_array_equal(rows(env), draw(n, ep).astype(np.float32).astype(np.float64))


def test_dynamics_randomization_refusals():
    from rl_aerial_manipulator_b200._cabi import QuadsimError
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    from rl_aerial_manipulator_b200.rollout import FusedRollout
    with pytest.raises(QuadsimError, match="RK4 handles only"):
        make_env(64, "v2", precision="f64", integrator="lsoda", dynamics_randomization=DR)
    for bad in (dict(mass=1.0), dict(inertia=-0.1), dict(thrust=1.5), dict(wind=-1.0), dict(mass=float("nan"))):
        with pytest.raises(QuadsimError, match="need finite"):
            make_env(64, "v2", dynamics_randomization=bad)
    env = make_env(64, "v2", precision="f32", dynamics_randomization=DR)
    env.reset()
    pol = MlpPolicyKernel.from_npz(os.path.join(os.path.dirname(__file__), "golden", "policy_v2.npz"), device="cuda", impl="tensor")
    with pytest.raises(ValueError, match="no dynamics randomisation"):
        FusedRollout(env, pol)
    env.dynamics_randomization = None                 # past the Python check: the C-ABI refuses too
    with pytest.raises(QuadsimError, match="fused rollout kernel has no dynamics randomisation"):
        FusedRollout(env, pol, sample="mean").step()
    with pytest.raises(ValueError, match="must be > 0"):
        env.set_dynamics(mass_scale=0.0)
    with pytest.raises(ValueError, match="finite"):
        env.set_dynamics(wind=float("inf"))
    with pytest.raises(ValueError, match="expected shape"):
        env.set_dynamics(thrust_scale=torch.ones(64, 3))
    env.randomize_dynamics(None)
    with pytest.raises(QuadsimError, match="not armed"):
        env.dynamics()
