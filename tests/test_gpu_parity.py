"""GPU parity tests: the sm_100a kernels, called through the C-ABI (libquadsim.so), against
  (a) the golden vectors produced by the unmodified reference (tests/golden/*.npz), and
  (b) the CPU oracle (oracle/quad_oracle.py) on identical seeded inputs.

Tolerances are BASELINE.json's north_star: float64 single step 1e-9 relative (LSODA parity mode vs the
reference), float32 1e-4, done/reset flags bit-exact, stated multi-step drift bound; the fixed-step float64
mode is checked at 1e-12 against the oracle's RK4 ("Oracle B").
"""
import os

import numpy as np
import pytest
import torch

from oracle import quad_oracle as qo

pytestmark = pytest.mark.gpu

VERS = {"v2": 2, "v1": 1, "v1_raw": 1, "v2m": 2}   # v2m: v2 with 2-3 waypoints (rl_env_scaledObs.py:46 alternative), ENV_V2M kernels
GOLDEN_OF = {"v2m": "v2"}


def make_env(n, variant="v2", **kw):
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    kw.setdefault("obs_scaled", variant != "v1_raw")
    if variant == "v2m":
        kw["v2_random_waypoints"] = True
    return BatchedQuadEnv(n, env_version=VERS[variant], **kw)


def load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def golden_select(g, variant):
    """Indices of golden cases the kernel layout can hold (v2 keeps one waypoint, like the shipped reference)."""
    idx = np.arange(len(g["reward"]))
    if variant == "v2":
        idx = idx[g["pre_n_wp"] == 1]
    return idx


def inject_golden(env, g, idx, prefix="pre_"):
    env.reset()
    env.set_state(y=g[prefix + "y"][idx], wp_list=g[prefix + "wp_list"][idx], n_wp=g[prefix + "n_wp"][idx].astype(np.int32),
                  wp_index=g[prefix + "wp_index"][idx].astype(np.int32), last_distance=g[prefix + "last_distance"][idx],
                  current_step=g[prefix + "current_step"][idx].astype(np.int32), counter=g[prefix + "counter"][idx].astype(np.int32),
                  final_reached=g[prefix + "final_reached"][idx].astype(np.uint8), final_yaw=g[prefix + "final_yaw"][idx],
                  ep_return=np.zeros(len(idx)), episode=np.zeros(len(idx), dtype=np.int32))


def golden_flags(g, idx):
    info = g["info"][idx].astype(np.int64)
    return (g["terminated"][idx].astype(np.int64) | (g["truncated"][idx].astype(np.int64) << 1) | ((info & 0xF) << 2)).astype(np.uint8)


def t2n(t):
    return t.detach().cpu().numpy()


# ------------------------------------------------------------------------------------------------------
# (a) golden vectors of the unmodified reference
# ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["v2", "v1", "v1_raw", "v2m"])
def test_f64_lsoda_single_step_vs_reference(golden_dir, variant):
    """float64 + LSODA port: state, obs and reward within 1e-9 of the reference's step; flags bit-exact.
    v2m runs ALL v2 cases, including the reference's multi-waypoint lists (2 and 3 entries), on the ENV_V2M kernels."""
    g = load(golden_dir, f"step_{GOLDEN_OF.get(variant, variant)}.npz")
    idx = golden_select(g, variant)
    env = make_env(len(idx), variant, precision="f64", integrator="lsoda", auto_reset=False)
    inject_golden(env, g, idx)
    out = env.step(torch.from_numpy(g["action"][idx]).cuda())
    st = {k: t2n(v) for k, v in env.get_state().items()}
    cnt, stp = env.lsoda_stats()
    cnt, stp = t2n(cnt), t2n(stp)
    ok = g["case"][idx] != "on_waypoint_nan"   # measure-zero case (distance exactly 0), covered by the logic test below

    np.testing.assert_allclose(st["y"], g["post_y"][idx], rtol=1e-9, atol=1e-10)
    np.testing.assert_array_equal(st["wp_index"], g["post_wp_index"][idx])
    np.testing.assert_array_equal(st["current_step"], g["post_current_step"][idx])
    if variant in ("v2", "v2m"):
        np.testing.assert_array_equal(st["counter"], g["post_counter"][idx])
        np.testing.assert_array_equal(st["final_reached"], g["post_final_reached"][idx].astype(np.uint8))
    np.testing.assert_allclose(st["last_distance"], g["post_last_distance"][idx], rtol=1e-9, atol=1e-10)
    np.testing.assert_array_equal(t2n(out.flags)[ok], golden_flags(g, idx)[ok])
    np.testing.assert_allclose(t2n(out.reward)[ok], g["reward"][idx][ok], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(t2n(out.obs), g["obs"][idx], rtol=3e-7, atol=1e-9)  # float32 obs: 1 ulp
    # the integrator walked the same step/order sequence as scipy's LSODA
    assert np.all(cnt[:, 3] == 0), "LSODA status flags raised"
    same = (cnt[:, 0] == g["lsoda_nst"][idx]) & (cnt[:, 1] == g["lsoda_nfe"][idx]) & (cnt[:, 2] == g["lsoda_nqu"][idx])
    assert same.mean() >= 0.98, f"only {same.sum()}/{len(idx)} calls reproduce scipy's (nst, nfe, nqu)"
    env.close()


@pytest.mark.parametrize("variant", ["v2", "v1", "v2m"])
def test_f32_rk4_single_step_vs_reference(golden_dir, variant):
    """float32 throughput mode vs the float64 reference: 1e-4 relative; flags equal."""
    g = load(golden_dir, f"step_{GOLDEN_OF.get(variant, variant)}.npz")
    idx = golden_select(g, variant)
    idx = idx[g["case"][idx] != "on_waypoint_nan"]
    env = make_env(len(idx), variant, precision="f32", integrator="rk4", substeps=1, auto_reset=False)
    inject_golden(env, g, idx)
    out = env.step(torch.from_numpy(g["action"][idx]).cuda())
    st = {k: t2n(v) for k, v in env.get_state().items()}
    np.testing.assert_allclose(st["y"], g["post_y"][idx], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(t2n(out.obs), g["obs"][idx], rtol=1e-4, atol=1e-5)
    np.testing.assert_array_equal(t2n(out.flags), golden_flags(g, idx))
    # the +2 progress bonus flips when |delta distance| is below float32 resolution: skip those rows
    ld, d = g["pre_last_distance"][idx], g["post_last_distance"][idx]
    ok = np.isnan(ld) | (np.abs(ld - d) >= 2e-6)
    np.testing.assert_allclose(t2n(out.reward)[ok], g["reward"][idx][ok], rtol=1e-4, atol=2e-4)
    assert ok.mean() > 0.95
    env.close()


@pytest.mark.parametrize("variant", ["v2", "v1"])
def test_seed0_and_trajectory_drift_vs_reference(golden_dir, variant):
    """Fixed-action multi-step trajectories of the reference (hover / random / controller actions, 600 steps):
    LSODA mode stays within the stated drift bound, flags bit-exact, auto-reset included."""
    g = load(golden_dir, f"traj_{variant}.npz")
    n_steps, n_env = g["action"].shape[:2]
    env = make_env(n_env, variant, precision="f64", integrator="lsoda", auto_reset=False)
    # start every env from the reference's own reset (golden uniforms are scripted, not Philox): inject via oracle
    b = qo.EnvBatch.empty(variant, n_env, max_wp=3)
    qo.reset_from_uniforms(b, np.arange(n_env), g["uniforms"][:, 0])
    episode = np.zeros(n_env, dtype=np.int64)

    def push(b):
        env.set_state(y=b.y, wp_list=b.wp_list, n_wp=b.n_wp.astype(np.int32), wp_index=b.wp_index.astype(np.int32),
                      last_distance=b.last_distance, current_step=b.current_step.astype(np.int32), counter=b.counter.astype(np.int32),
                      final_reached=b.final_reached.astype(np.uint8), final_yaw=b.final_yaw)
    env.reset()
    push(b)
    worst_r = worst_o = 0.0
    for t in range(n_steps):
        out = env.step(torch.from_numpy(g["action"][t]).cuda())
        flags = t2n(out.flags)
        want = g["terminated"][t].astype(np.uint8) | (g["truncated"][t].astype(np.uint8) << 1) | ((g["info"][t] & 0xF) << 2)
        np.testing.assert_array_equal(flags, want, err_msg=f"t={t}")
        worst_r = max(worst_r, np.abs(t2n(out.reward) - g["reward"][t]).max())
        worst_o = max(worst_o, np.abs(t2n(out.obs).astype(np.float64) - g["terminal_obs"][t]).max())
        done = (flags & 3) != 0
        if done.any():   # replay the reference's scripted reset for the finished envs
            st = {k: t2n(v) for k, v in env.get_state().items()}
            for f in ("y", "wp_list", "n_wp", "wp_index", "last_distance", "current_step", "counter", "final_yaw"):
                setattr(b, f, st[f].astype(getattr(b, f).dtype))
            b.final_reached = st["final_reached"].astype(bool)
            ids = np.nonzero(done)[0]
            episode[ids] += 1
            qo.reset_from_uniforms(b, ids, g["uniforms"][ids, episode[ids]])
            push(b)
    # drift bound stated in DESIGN.md: 2e-6 on reward (it carries 20*delta-distance), 1e-6 on obs over 600 steps
    assert worst_r < 2e-6 and worst_o < 1e-6, (worst_r, worst_o)
    assert (g["terminated"] | g["truncated"]).sum() >= 3
    env.close()


# ------------------------------------------------------------------------------------------------------
# (b) the oracle on identical seeded inputs
# ------------------------------------------------------------------------------------------------------
def random_batch(variant, n, seed):
    rng = np.random.default_rng(seed)
    b = qo.EnvBatch.empty(variant, n, max_wp=3)
    b.y[:, 0:3] = rng.uniform(-2, 2, (n, 3))
    b.y[:, 2] = rng.uniform(0.05, 3.0, n)
    b.y[:, 3:6] = rng.normal(size=(n, 3))
    q = rng.normal(size=(n, 4)) * rng.choice([0.05, 0.5, 2.0], size=(n, 1)) + [1, 0, 0, 0]
    b.y[:, 6:10] = q / np.linalg.norm(q, axis=1, keepdims=True)
    b.y[:, 10:13] = rng.normal(size=(n, 3)) * 2
    k = 1 if variant == "v2" else 2
    b.n_wp[:] = 1 if variant == "v2" else rng.integers(1, 3, n)
    b.wp_list[:, :k] = np.stack([rng.uniform(-1, 1, (n, k)), rng.uniform(-1, 1, (n, k)), rng.uniform(1, 3, (n, k))], -1)
    near = rng.random(n) < 0.3           # a third of the envs sit close to their waypoint
    b.wp_index[:] = 0
    b.cur_wp = b.wp_list[:, 0].copy()
    b.y[near, 0:3] = b.cur_wp[near] + rng.normal(size=(near.sum(), 3)) * 0.06
    b.y[near, 3:6] *= 0.05
    d = np.linalg.norm(b.y[:, 0:3] - b.cur_wp, axis=1)
    b.last_distance = np.where(rng.random(n) < 0.1, np.nan, d + rng.normal(size=n) * 0.01)
    b.current_step = rng.integers(0, 2003 if variant == "v2" else 1203, n)
    if variant == "v2":
        fin = near & (rng.random(n) < 0.5)
        b.final_reached = fin
        b.wp_index = np.where(fin, 1, 0)
        b.counter = np.where(fin, rng.integers(0, 520, n), 0)
        b.final_yaw = rng.uniform(-np.pi, np.pi, n)
    a = np.stack([rng.uniform(0, 2, n), *rng.uniform(-1, 1, (3, n))], 1).astype(np.float32)
    return b, a


def push_batch(env, b):
    env.reset()
    env.set_state(y=b.y, wp_list=b.wp_list, n_wp=b.n_wp.astype(np.int32), wp_index=b.wp_index.astype(np.int32),
                  last_distance=b.last_distance, current_step=b.current_step.astype(np.int32), counter=b.counter.astype(np.int32),
                  final_reached=b.final_reached.astype(np.uint8), final_yaw=b.final_yaw,
                  ep_return=np.zeros(b.n), episode=np.zeros(b.n, dtype=np.int32))


@pytest.mark.parametrize("variant,substeps", [("v2", 1), ("v2", 4), ("v1", 1), ("v1_raw", 2)])
def test_f64_rk4_vs_oracle_65536(variant, substeps):
    """config 3 size: 65,536 envs, float64 fixed-step mode vs the oracle's RK4 at 1e-12; flags bit-exact."""
    n = 65536
    b, a = random_batch(variant, n, seed=11)
    env = make_env(n, variant, precision="f64", integrator="rk4", substeps=substeps, auto_reset=False)
    push_batch(env, b)
    out = env.step(torch.from_numpy(a).cuda())
    with np.errstate(all="ignore"):
        obs, rew, term, trunc, info = qo.step(b, a, integrator="rk4", substeps=substeps)
    st = {k: t2n(v) for k, v in env.get_state().items()}
    np.testing.assert_allclose(st["y"], b.y, rtol=1e-12, atol=1e-13)
    want = term.astype(np.uint8) | (trunc.astype(np.uint8) << 1) | ((info & 0xF) << 2)
    flags = t2n(out.flags)
    # a threshold compare (d < 0.1, z < 0.1 ...) may flip when the two float64 results straddle it by 1 ulp
    assert (flags != want).sum() <= 2
    same = flags == want
    np.testing.assert_allclose(t2n(out.reward)[same], rew[same], rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(t2n(out.obs)[same], obs[same], rtol=2e-7, atol=1e-12)
    np.testing.assert_array_equal(st["counter"][same], b.counter[same])
    np.testing.assert_array_equal(st["current_step"][same], b.current_step[same])
    np.testing.assert_array_equal(st["wp_index"][same], b.wp_index[same])
    env.close()


@pytest.mark.parametrize("variant", ["v2", "v1"])
def test_f32_rk4_vs_oracle_65536(variant):
    n = 65536
    b, a = random_batch(variant, n, seed=12)
    env = make_env(n, variant, precision="f32", integrator="rk4", substeps=1, auto_reset=False)
    push_batch(env, b)
    out = env.step(torch.from_numpy(a).cuda())
    with np.errstate(all="ignore"):
        obs, rew, term, trunc, info = qo.step(b, a, integrator="rk4", substeps=1)
    st = {k: t2n(v) for k, v in env.get_state().items()}
    np.testing.assert_allclose(st["y"], b.y, rtol=1e-4, atol=1e-5)
    want = term.astype(np.uint8) | (trunc.astype(np.uint8) << 1) | ((info & 0xF) << 2)
    flags = t2n(out.flags)
    assert (flags != want).mean() < 2e-4          # float32 rounding next to a threshold
    same = flags == want
    ld, d = t2n(env.get_state(["last_distance"])["last_distance"]), b.last_distance
    np.testing.assert_allclose(t2n(out.obs)[same], obs[same], rtol=1e-4, atol=1e-5)
    rel = np.abs(t2n(out.reward)[same].astype(np.float64) - rew[same]) / np.maximum(np.abs(rew[same]), 1.0)
    assert np.mean(rel < 1e-4) > 0.999            # the rest: +2 progress bonus flipped by float32 resolution
    env.close()


@pytest.mark.parametrize("variant", ["v2", "v1", "v2m"])
def test_reset_matches_oracle_on_device_uniforms(variant):
    """Reset sampling: the kernel's Philox uniforms, replayed through the (reference-pinned) oracle reset."""
    n = 4099  # ragged: not a multiple of the warp or block size
    env = make_env(n, variant, precision="f64", integrator="rk4", seed=77, env_id_offset=5_000_000_000)
    obs = t2n(env.reset()).copy()
    ids = torch.arange(n, dtype=torch.int64) + 5_000_000_000
    U = t2n(env.reset_uniforms(ids, torch.zeros(n, dtype=torch.int32)))
    assert U.min() >= 0 and U.max() < 1 and abs(U.mean() - 0.5) < 0.01
    b = qo.EnvBatch.empty(GOLDEN_OF.get(variant, variant), n, max_wp=3)
    b.v2_random_waypoints = variant == "v2m"
    qo.reset_from_uniforms(b, np.arange(n), U)
    st = {k: t2n(v) for k, v in env.get_state().items()}
    np.testing.assert_array_equal(st["y"], b.y)
    k = {"v2": 1, "v1": 2, "v2m": 3}[variant]
    np.testing.assert_array_equal(st["wp_list"][:, :k], b.wp_list[:, :k])
    np.testing.assert_array_equal(st["n_wp"], b.n_wp)
    if variant == "v2m":
        assert set(np.unique(st["n_wp"])) == {2, 3}
    assert np.all(np.isnan(st["last_distance"])) and np.all(st["current_step"] == 0) and np.all(st["episode"] == 0)
    if variant in ("v2", "v2m"):
        np.testing.assert_array_equal(st["final_yaw"], b.final_yaw)
    np.testing.assert_array_equal(obs, qo.observe(b))
    # masked reset touches only the masked envs and advances their episode counter
    mask = torch.zeros(n, dtype=torch.uint8)
    mask[::7] = 1
    env.reset(mask)
    st2 = {k: t2n(v) for k, v in env.get_state(["y", "episode"]).items()}
    m = t2n(mask).astype(bool)
    assert np.all(st2["episode"][m] == 1) and np.all(st2["episode"][~m] == 0)
    np.testing.assert_array_equal(st2["y"][~m], st["y"][~m])
    assert np.all(np.any(st2["y"][m] != st["y"][m], axis=1))
    env.close()


@pytest.mark.parametrize("variant", ["v2", "v1", "v2m"])
def test_vec_rollout_with_autoreset_vs_oracle(variant):
    """N envs, random actions, auto-reset inside the kernel: the oracle (scipy LSODA) driven by the very same
    Philox uniforms must see the same dones, terminal observations, episode returns/lengths and next obs."""
    n, steps = 48, 160
    env = make_env(n, variant, precision="f64", integrator="lsoda", seed=5)
    seed_ids = torch.arange(n, dtype=torch.int64)

    def uniforms(ids, eps):
        return t2n(env.reset_uniforms(torch.as_tensor(ids, dtype=torch.int64), torch.as_tensor(eps, dtype=torch.int32)))

    vec = qo.VecOracle(GOLDEN_OF.get(variant, variant), n, uniforms, integrator="lsoda", max_wp=3, v2_random_waypoints=(variant == "v2m"))
    obs_o = vec.reset()
    obs_k = t2n(env.reset()).copy()
    np.testing.assert_array_equal(obs_k, obs_o)
    rng = np.random.default_rng(3)
    n_done = 0
    for t in range(steps):
        a = np.stack([rng.uniform(0, 2, n), *rng.uniform(-1, 1, (3, n))], 1).astype(np.float32)
        if t % 3 == 0:
            a[: n // 2] = [0.2, 0, 0, 0]    # half the envs drop to the ground -> crashes and resets
        out = env.step(torch.from_numpy(a).cuda())
        with np.errstate(all="ignore"):
            obs_o, rew_o, done_o, ex = vec.step(a)
        flags = t2n(out.flags)
        want = ex["terminated"].astype(np.uint8) | (ex["truncated"].astype(np.uint8) << 1) | ((ex["info"] & 0xF) << 2)
        np.testing.assert_array_equal(flags, want, err_msg=f"t={t}")
        np.testing.assert_allclose(t2n(out.reward), rew_o, rtol=0, atol=2e-6)
        np.testing.assert_allclose(t2n(out.obs), obs_o, rtol=0, atol=1e-6)
        d = done_o
        if d.any():
            n_done += d.sum()
            np.testing.assert_allclose(t2n(out.terminal_obs)[d], ex["terminal_obs"][d], rtol=0, atol=1e-6)
            np.testing.assert_allclose(t2n(out.ep_return)[d], ex["ep_return"][d], rtol=1e-8, atol=1e-5)
            np.testing.assert_array_equal(t2n(out.ep_len)[d], ex["ep_len"][d])
    assert n_done >= 20
    env.close()


# ------------------------------------------------------------------------------------------------------
# (c) full-size, size-independent properties
# ------------------------------------------------------------------------------------------------------
def test_properties_1M_envs_f32():
    """config 4/5 shard size (1,048,576 envs, float32): invariants that need no oracle."""
    n = 1 << 20
    env = make_env(n, "v2", precision="f32", seed=9)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    lo = torch.tensor([0.0, -1, -1, -1], device="cuda")
    hi = torch.tensor([2.0, 1, 1, 1], device="cuda")
    ep_done = torch.zeros(n, dtype=torch.int64, device="cuda")
    n_steps = 200
    for t in range(n_steps):
        a = lo + (hi - lo) * torch.rand((n, 4), device="cuda", generator=g)
        a[: n // 2, 0] *= 0.25                                      # half the envs sink and crash -> auto-reset
        out = env.step(a)
        ep_done += out.done
        assert torch.isfinite(out.obs).all() and torch.isfinite(out.reward).all()
        q = out.obs[:, 6:10].double()
        assert (q.norm(dim=1) - 1).abs().max() < 1e-6            # renormalised every step (quadcopter.py:114)
    st = env.get_state(["episode", "current_step", "y"])
    assert torch.equal(st["episode"].long(), ep_done)              # one reset per done, nothing else resets
    assert int(ep_done.sum()) > 0
    assert int(ep_done[: n // 2].sum()) > n // 4
    assert (st["current_step"] <= n_steps).all() and (st["y"][:, 2] > -1).all()
    env.close()


def test_config5_total_size_on_one_gpu_matches_small_batches():
    """8,388,608 envs (BASELINE configs[4] total) in one handle: 64-bit addressing of the pool and obs, and the same episodes as
    small handles placed at the head, in the middle and at the tail of the global env-id range (Philox keyed on the global id)."""
    n = 8 * (1 << 20)
    big = make_env(n, "v2", precision="f32", seed=4)
    big.reset()
    g = torch.Generator(device="cuda").manual_seed(1)
    acts = [(torch.rand((n, 4), device="cuda", generator=g) * torch.tensor([0.7, 2, 2, 2], device="cuda")
             - torch.tensor([0, 1, 1, 1.0], device="cuda")) for _ in range(2)]
    small = {}
    m = 4096
    for off in (0, n // 2 + 31, n - m):
        from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
        small[off] = BatchedQuadEnv(m, env_version=2, precision="f32", seed=4, env_id_offset=off)
        small[off].reset()
    for t in range(120):
        a = acts[t & 1]
        out = big.step(a)
        for off, env in small.items():
            o = env.step(a[off:off + m].contiguous())
            assert torch.equal(o.obs, out.obs[off:off + m]) and torch.equal(o.flags, out.flags[off:off + m]), (t, off)
            assert torch.equal(o.reward, out.reward[off:off + m])
    assert torch.isfinite(out.obs).all()
    assert int((big.get_state(["episode"])["episode"] > 0).sum()) > n // 10      # low thrust: many crash and reset
    big.close()
    for env in small.values():
        env.close()


def test_determinism_and_shard_independence():
    """Same seed -> same rollout; a batch split over two handles with env_id_offset draws the same episodes."""
    n, steps = 8192, 200
    g = torch.Generator(device="cuda").manual_seed(1)
    acts = [torch.rand((n, 4), device="cuda", generator=g) * torch.tensor([0.6, 2, 2, 2], device="cuda") - torch.tensor([0.0, 1, 1, 1], device="cuda")
            for _ in range(steps)]   # low thrust: every env crashes and is auto-reset at least once

    def run(n_envs, offset, sl):
        env = make_env(n_envs, "v2", precision="f32", seed=21, env_id_offset=offset)
        env.reset()
        rews, dones = [], []
        for a in acts:
            out = env.step(a[sl].contiguous())
            rews.append(out.reward.clone())
            dones.append(out.done.clone())
        obs = out.obs.clone()
        env.close()
        return torch.stack(rews), torch.stack(dones), obs

    full = run(n, 0, slice(0, n))
    again = run(n, 0, slice(0, n))
    for x, y in zip(full, again):
        assert torch.equal(x, y)
    lo = run(n // 2, 0, slice(0, n // 2))
    hi = run(n // 2, n // 2, slice(n // 2, n))
    assert torch.equal(torch.cat([lo[0], hi[0]], 1), full[0])
    assert torch.equal(torch.cat([lo[1], hi[1]], 1), full[1])
    assert torch.equal(torch.cat([lo[2], hi[2]], 0), full[2])
    assert int(full[1].sum()) > n // 2


@pytest.mark.parametrize("n", [1, 31, 33, 257])
def test_ragged_batch_sizes(n):
    env = make_env(n, "v2", precision="f32", seed=2)
    big = make_env(1024, "v2", precision="f32", seed=2)
    o1, o2 = env.reset().clone(), big.reset().clone()
    assert torch.equal(o1, o2[:n])
    a = torch.rand((1024, 4), device="cuda")
    r1 = env.step(a[:n].contiguous())
    r2 = big.step(a)
    assert torch.equal(r1.obs, r2.obs[:n]) and torch.equal(r1.reward, r2.reward[:n]) and torch.equal(r1.flags, r2.flags[:n])
    env.close()
    big.close()


def test_error_paths():
    from rl_aerial_manipulator_b200 import QuadsimError
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    with pytest.raises(QuadsimError):
        BatchedQuadEnv(8, precision="f32", integrator="lsoda")      # LSODA needs float64
    with pytest.raises(QuadsimError):
        BatchedQuadEnv(0)
    env = BatchedQuadEnv(8)
    with pytest.raises(QuadsimError):
        env.step(torch.zeros((8, 4), device="cuda"))                  # step before reset
    env.reset()
    with pytest.raises(ValueError):
        env.step(torch.zeros((8, 3), device="cuda"))
    env.close()


# ------------------------------------------------------------------------------------------------------
# (d) the SB3 VecEnv surface (NumPy in/out, infos) against the oracle's DummyVecEnv/Monitor restatement
# ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant,info_mode", [("v2", "dict"), ("v1", "lazy")])
def test_quad_vec_env_surface_vs_oracle(variant, info_mode):
    from rl_aerial_manipulator_b200.vec_env import QuadVecEnv
    n, steps = 32, 260
    venv = QuadVecEnv(n, env_version=VERS[variant], precision="f64", integrator="lsoda", seed=8, info_mode=info_mode)
    assert venv.num_envs == n and venv.observation_space.shape == (20 if variant == "v2" else 17,)
    np.testing.assert_array_equal(venv.action_space.low, [0, -1, -1, -1])
    np.testing.assert_array_equal(venv.action_space.high, [2, 1, 1, 1])

    def uniforms(ids, eps):
        return t2n(venv.sim.reset_uniforms(torch.as_tensor(ids, dtype=torch.int64), torch.as_tensor(eps, dtype=torch.int32)))

    vec = qo.VecOracle(variant, n, uniforms, integrator="lsoda", max_wp=3)
    obs = venv.reset()
    assert obs.dtype == np.float32 and obs.shape == (n, venv.sim.obs_dim)
    np.testing.assert_array_equal(obs, vec.reset())
    rng = np.random.default_rng(5)
    seen = {"crashed": 0, "episode": 0, "trunc_key": 0}
    for t in range(steps):
        a = np.stack([rng.uniform(0, 0.3, n), *rng.uniform(-1, 1, (3, n))], 1).astype(np.float32)
        venv.step_async(a)
        obs, rew, dones, infos = venv.step_wait()
        with np.errstate(all="ignore"):
            obs_o, rew_o, done_o, ex = vec.step(a)
        assert rew.dtype == np.float32 and dones.dtype == np.bool_ and len(infos) == n
        np.testing.assert_array_equal(dones, done_o)
        np.testing.assert_allclose(obs, obs_o, rtol=0, atol=1e-6)
        np.testing.assert_allclose(rew, rew_o.astype(np.float32), rtol=1e-6, atol=1e-5)
        for i in range(n):
            info = infos[i]
            if not dones[i]:
                assert "terminal_observation" not in info and "episode" not in info
                continue
            # DummyVecEnv: terminal_observation + TimeLimit.truncated; Monitor: episode r / l
            np.testing.assert_allclose(info["terminal_observation"], ex["terminal_obs"][i], rtol=0, atol=1e-6)
            assert info["TimeLimit.truncated"] == bool(ex["truncated"][i] and not ex["terminated"][i])
            assert info["episode"]["l"] == ex["ep_len"][i] and abs(info["episode"]["r"] - ex["ep_return"][i]) < 1e-4
            bits = int(ex["info"][i])
            assert info.get("crashed", False) == bool(bits & qo.INFO_CRASHED)
            assert info.get("out_of_bounds", False) == bool(bits & qo.INFO_OOB)
            if bits & (qo.INFO_CRASHED | qo.INFO_OOB):
                assert info["success"] is False
            seen["crashed"] += bool(bits & qo.INFO_CRASHED)
            seen["episode"] += 1
    assert seen["episode"] >= n and seen["crashed"] >= n // 2
    st = venv.get_attr("waypoint_list", [0, 1])
    assert len(st) == 2 and st[0][0].shape == (3,)
    assert venv.env_is_wrapped(object) == [False] * n and venv.seed() == [8] * n
    venv.close()


# ------------------------------------------------------------------------------------------------------
# (e) BASELINE.json configs[0] / configs[1]: the reference's own CPU-runnable cases, on the GPU path
# ------------------------------------------------------------------------------------------------------
def test_config0_v1_hover_10k_steps():
    """configs[0]: v1 rl_env_scaledObs, one env, 10,000 steps of the fixed hover action float32 [1,0,0,0] with auto-reset.
    The reference truncates on the 1,201st step of an episode, so 10,000 steps contain exactly 8 resets (SURVEY appendix A);
    hovering keeps the vehicle within millimetres of its start."""
    env = make_env(1, "v1", precision="f64", integrator="lsoda", seed=0)
    obs0 = env.reset().clone()
    a = torch.tensor([[1.0, 0, 0, 0]], device="cuda")
    dones, truncs, terms = 0, 0, 0
    lens = []
    for t in range(10000):
        out = env.step(a)
        f = int(out.flags[0])
        if f & 3:
            dones += 1
            truncs += bool(f & 2)
            terms += bool(f & 1)
            lens.append(int(out.ep_len[0]))
    assert dones == 8 and truncs == 8 and terms == 0 and lens == [1201] * 8
    st = env.get_state(["current_step", "episode", "y"])
    assert int(st["episode"][0]) == 8 and int(st["current_step"][0]) == 10000 - 8 * 1201
    # F = fl32(fl32(1*fl32(0.18))*fl32(9.81)) = 1.7658001 N vs m*g = 1.7658 N: the hover drifts by < 1 mm per episode
    assert abs(float(st["y"][0, 5])) < 1e-3
    env.close()


@pytest.mark.parametrize("precision,integrator", [("f64", "lsoda"), ("f32", "rk4")])
def test_config1_shipped_v1_policy_flies_the_course(golden_dir, precision, integrator):
    """configs[1]-style closed loop: the reference's shipped v1 policy (waypoint_controller_scaledObs_4M.zip, deterministic
    actions, SB3-style clipping) drives 512 GPU envs.  On the reference env it reaches every waypoint (SURVEY section 4:
    6/6 episodes, 252-508 steps, return 2362-5221); the GPU env must give the same picture."""
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    n = 512
    env = make_env(n, "v1", precision=precision, integrator=integrator, seed=3)
    pol = MlpPolicyKernel.from_npz(os.path.join(golden_dir, "policy_v1.npz"), device="cuda", impl="fp32")
    obs = env.reset()
    n_success, n_other, lens, rets = 0, 0, [], []
    for t in range(700):
        pol.forward(obs)                               # deterministic: the mean action
        out = env.step(pol.actions_clipped)
        obs = out.obs
        flags = t2n(out.flags)
        d = (flags & 3) != 0
        if d.any():
            succ = d & ((flags & 4) != 0)
            n_success += int(succ.sum())
            n_other += int((d & ~succ).sum())
            lens += t2n(out.ep_len)[succ].tolist()
            rets += t2n(out.ep_return)[succ].tolist()
    assert n_success >= n and n_other <= 0.02 * (n_success + n_other), (n_success, n_other)
    assert 30 <= np.min(lens) and np.max(lens) <= 800 and 200 <= np.median(lens) <= 520, (np.min(lens), np.median(lens), np.max(lens))
    assert 1500 <= np.median(rets) <= 6000
    env.close()


def test_chunked_host_pipeline_equals_single_launch(golden_dir):
    """QuadVecEnv(pipeline_chunks=4) (qs_step_range on four streams) and predict_host(pipeline_chunks=4) return exactly what the
    single-launch paths return: sub-ranges of whole warp tiles are independent."""
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    from rl_aerial_manipulator_b200.vec_env import QuadVecEnv
    n = 10_000 + 37                                              # ragged: last chunk and last tile partially filled
    a = QuadVecEnv(n, env_version=2, seed=8, pipeline_chunks=1, info_mode="lazy")
    b = QuadVecEnv(n, env_version=2, seed=8, pipeline_chunks=4, info_mode="lazy")
    assert len(b._chunks) == 4 and all(f % 32 == 0 for f, _ in b._chunks) and sum(c for _, c in b._chunks) == n
    oa, ob = a.reset(), b.reset()
    np.testing.assert_array_equal(oa, ob)
    rng = np.random.default_rng(0)
    pol = MlpPolicyKernel.from_npz(os.path.join(golden_dir, "policy_v2.npz"), device="cuda", impl="tensor")
    for t in range(160):
        act = (np.array([0, -1, -1, -1.0]) + np.array([0.4, 2, 2, 2.0]) * rng.random((n, 4))).astype(np.float32)
        oa, ra, da, _ = a.step(act)
        ob, rb, db, _ = b.step(act)
        np.testing.assert_array_equal(oa, ob)
        np.testing.assert_array_equal(ra, rb)
        np.testing.assert_array_equal(da, db)
    assert da.sum() >= 0 and int(a.sim.get_state(["episode"])["episode"].sum()) > 0       # some envs crashed and were reset
    p1 = pol.predict_host(oa, stochastic=False, pipeline_chunks=1).copy()
    p4 = pol.predict_host(oa, stochastic=False, pipeline_chunks=4).copy()
    np.testing.assert_array_equal(p1, p4)
    a.close()
    b.close()


@pytest.mark.parametrize("n", [1, 31, 33, 1013, 4097])
def test_no_writes_past_the_batch_end(golden_dir, n):
    """Ragged batch sizes with guard rows behind every output buffer (the pool's sanitizer is not available): the step kernels,
    the reset kernel and the three policy kernels must leave the rows past n untouched."""
    from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
    guard = 96
    sentinel = 1234.5

    def guarded(shape, dtype):
        big = torch.full((shape[0] + guard, *shape[1:]), sentinel if dtype.is_floating_point else 77, dtype=dtype, device="cuda")
        return big, big[: shape[0]]

    for variant, prec in (("v2", "f32"), ("v1", "f32"), ("v2", "f64"), ("v2m", "f32")):
        env = make_env(n, variant, precision=prec, seed=3)
        bigs = {}
        for name in ("obs", "reward", "flags", "terminal_obs", "ep_return", "ep_len"):
            t = getattr(env, name)
            bigs[name], view = guarded(tuple(t.shape), t.dtype)
            setattr(env, name, view)
        env.reset()
        for t in range(3):
            env.step(torch.rand((n, 4), device="cuda"))
        for name, big in bigs.items():
            tail = big[n:]
            want = sentinel if big.dtype.is_floating_point else 77
            assert bool((tail == want).all()), (variant, prec, name)
        assert torch.isfinite(env.obs).all()
        env.close()
    for impl in ("fp32", "tensor", "tensor_fast"):
        pol = MlpPolicyKernel.from_npz(os.path.join(golden_dir, "policy_v2.npz"), device="cuda", impl=impl)
        pol._ensure(n)
        bigs = {}
        for name in ("actions", "actions_clipped", "values", "logp"):
            t = getattr(pol, name)
            bigs[name], view = guarded(tuple(t.shape), t.dtype)
            setattr(pol, name, view)
        obs = torch.randn((n, 20), device="cuda")
        big_norm, norm_out = guarded((n, 20), torch.float32)
        stats = torch.zeros(41, dtype=torch.float64, device="cuda"); stats[0] = 1.0; stats[21:] = 1.0
        pol.forward(obs, torch.randn((n, 4), device="cuda"), norm_stats=stats, obs_norm_out=norm_out)
        torch.cuda.synchronize()
        for name, big in {**bigs, "obs_norm_out": big_norm}.items():
            assert bool((big[n:] == sentinel).all()), (impl, name)
        assert torch.isfinite(pol.actions).all() and torch.isfinite(norm_out).all()
