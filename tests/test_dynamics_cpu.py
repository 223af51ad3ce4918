"""Dynamics randomisation on the CPU: the C-ABI struct layout, the per-episode draw of the device headers (compiled with g++)
against a NumPy Philox restatement, the oracle's randomised model against the nominal one and against closed-form single
steps, and the device headers' randomised step against the oracle on random states and random parameters."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import dyn_oracle as do
from oracle import quad_oracle as qo
from dyn_harness import DynHarness
from harness_util import ROOT


@pytest.fixture(scope="module")
def cabi():
    from rl_aerial_manipulator_b200 import _cabi
    return _cabi


@pytest.fixture(scope="module")
def hh(cabi):
    return DynHarness(cabi.make_config(env_version=2, seed=11))


def test_dynamics_rand_ctypes_layout_matches_header(cabi, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "quadsim.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %d\\n", sizeof(qs_dynamics_rand), offsetof(qs_dynamics_rand, seed),\n'
                   '         offsetof(qs_dynamics_rand, mass_rel), offsetof(qs_dynamics_rand, inertia_rel),\n'
                   '         offsetof(qs_dynamics_rand, thrust_rel), offsetof(qs_dynamics_rand, wind), QS_DYN_PARAMS);\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    R = cabi.QsDynamicsRand
    want = [C.sizeof(R)] + [getattr(R, f).offset for f in ("seed", "mass_rel", "inertia_rel", "thrust_rel", "wind")] + [cabi.DYN_PARAMS]
    assert got == want


def test_draw_equals_numpy_restatement_bitwise(hh):
    rng = np.random.default_rng(0)
    for seed, ranges in [(0, (0.3, 0.2, 0.1, 0.5)), (2**64 - 1, (0.999, 0.5, 1.0, 3.0)), (12345, (0.0, 0.0, 0.0, 0.0))]:
        gids = np.concatenate([np.arange(200), rng.integers(0, 2**40, 200), [2**32 - 1, 2**32, 2**63 - 1]]).astype(np.uint64)
        eps = rng.integers(0, 2**31, len(gids))
        want = do.dynamics_draw(seed, *ranges, gids, eps)
        got = np.stack([hh.dyn_draw(seed, ranges, int(g), int(e)) for g, e in zip(gids, eps)])
        np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64))
    d = do.dynamics_draw(7, 0.3, 0.2, 0.1, 0.5, np.arange(20000), np.zeros(20000))
    assert np.all(np.abs(d[:, 0] - 1) <= 0.3) and np.all(np.abs(d[:, 2:6] - 1) <= 0.1) and np.all(np.abs(d[:, 6:]) <= 0.5)
    np.testing.assert_allclose(d.mean(0), [1, 1, 1, 1, 1, 1, 0, 0, 0], atol=0.01)       # uniform, centred
    assert abs(np.corrcoef(d[:, 0], d[:, 2])[0, 1]) < 0.03                               # independent parameters


def test_draw_stream_independent_of_reset_stream(hh):
    """Counter word 3 of the draw (0x100 + b) never meets the reset's (j < 9): the same seed gives unrelated uniforms."""
    u_reset = hh.uniforms(5, 17, 3)
    d = hh.dyn_draw(5, (0.5, 0.5, 0.5, 1.0), 17, 3)
    u_dyn0 = (d[0] - 1) / 0.5 * 0.5 + 0.5
    assert not np.any(np.isclose(u_reset, u_dyn0, rtol=0, atol=1e-12))


def _random_y(rng, n):
    y = np.zeros((n, 13))
    y[:, 0:3] = rng.uniform(-2, 2, (n, 3)) + [0, 0, 2]
    y[:, 3:6] = rng.normal(size=(n, 3))
    q = rng.normal(size=(n, 4)) * 0.3 + [1, 0, 0, 0]
    y[:, 6:10] = q / np.linalg.norm(q, axis=1, keepdims=True)
    y[:, 10:13] = rng.normal(size=(n, 3)) * 1.5
    return y


def test_oracle_unit_factors_equal_nominal_bitwise():
    rng = np.random.default_rng(1)
    n = 2000
    y = _random_y(rng, n)
    act = np.stack([rng.uniform(0, 2, n), *rng.uniform(-1, 1, (3, n))], 1).astype(np.float32)
    nominal = qo.physics_update(y, act, "rk4", substeps=2)
    unit = do.physics_update(y, act, substeps=2, mass_scale=np.ones(n), inertia_scale=np.ones(n), thrust_scale=np.ones((n, 4)),
                             wind=np.zeros((n, 3)))
    np.testing.assert_array_equal(unit.view(np.uint64), nominal.view(np.uint64))


def _hover(n=1):
    y = np.zeros((n, 13))
    y[:, 2] = 2.0
    y[:, 6] = 1.0
    return y


@pytest.mark.parametrize("k", [0.7, 0.9, 1.0, 1.25, 1.6])
def test_hover_with_mass_factor(k):
    """Hover action (commands the nominal m*g) on an airframe of mass m*k: one step from rest changes vz by g(1/k - 1) dt."""
    y = _hover()
    y2 = do.physics_update(y, np.array([[1.0, 0, 0, 0]]), action_f32=False, mass_scale=np.array([k]))
    np.testing.assert_allclose(y2[0, 5], qo.GRAV * (1 / k - 1) * qo.DT, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(y2[0, [3, 4, 10, 11, 12]], 0, atol=1e-15)


def test_wind_only():
    """Hover on the nominal airframe with a wind force f: dv = f / (m k_m) dt."""
    f = np.array([[0.3, -0.2, 0.1], [-1.0, 0.5, 0.0]])
    km = np.array([1.0, 1.3])
    y2 = do.physics_update(_hover(2), np.array([[1.0, 0, 0, 0]] * 2), action_f32=False, mass_scale=km, wind=f)
    want = f / (qo.MASS * km)[:, None] * qo.DT
    want[:, 2] += qo.GRAV * (1 / km - 1) * qo.DT           # the second env is also heavier than the hover command assumes
    np.testing.assert_allclose(y2[:, 3:6], want, rtol=1e-12, atol=1e-15)


def test_yaw_command_scales_with_inverse_inertia():
    """Hover plus a small yaw command (every prop inside the clamp): the body-rate change after one step scales as 1/k_I."""
    a = np.array([[1.0, 0, 0, 0.05]], dtype=np.float64)
    _, _, t = qo.mix_and_clamp(*qo.scale_action(a, False))
    assert np.all((t > qo.MIN_F / 4) & (t < qo.MAX_F / 4))
    w1 = qo.physics_update(_hover(), a, "rk4", action_f32=False)[0, 10:13]
    assert abs(w1[2]) > 1e-3
    for kI in (0.6, 0.8, 1.2, 1.5):
        wk = do.physics_update(_hover(), a, action_f32=False, inertia_scale=np.array([kI]))[0, 10:13]
        # first order in dt: J M dt / k_I; the gyroscopic term w x (k_I I w) inside the step adds ~1e-7 rad/s to the pitch rate
        np.testing.assert_allclose(wk, w1 / kI, rtol=1e-6, atol=1e-6)


def _random_batch(rng, variant, n):
    """Random internal states around every threshold of the step logic (the scheme of test_randomised_states_step_matches_oracle)."""
    oname = "v1" if variant == "v1" else "v2"
    kmax = {"v2": 1, "v1": 2, "v2m": 3}[variant]
    b = qo.EnvBatch.empty(oname, n, max_wp=3)
    b.n_wp[:] = rng.integers(1, kmax + 1, n)
    b.wp_list[:] = np.stack([rng.uniform(-1, 1, (n, 3)), rng.uniform(-1, 1, (n, 3)), rng.uniform(0.3, 3, (n, 3))], -1)
    b.wp_index[:] = np.clip(np.minimum(rng.integers(0, 3, n), b.n_wp - (rng.random(n) < 0.5)), 0, b.n_wp)
    ar = np.arange(n)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    r = np.where(rng.random(n) < 0.35, rng.uniform(0.09, 0.11, n), rng.uniform(0.0, 2.5, n))
    b.cur_wp = b.wp_list[ar, np.minimum(b.wp_index, b.n_wp - 1)].copy()
    b.y[:] = 0
    b.y[:, 0:3] = b.cur_wp + d * r[:, None]
    low = rng.random(n) < 0.08
    b.y[low, 2] = rng.uniform(0.09, 0.11, low.sum())
    b.y[:, 3:6] = rng.normal(size=(n, 3)) * np.where(rng.random(n) < 0.3, 0.05, 1.0)[:, None]
    q = rng.normal(size=(n, 4)) * 0.3 + [1, 0, 0, 0]
    b.y[:, 6:10] = q / np.linalg.norm(q, axis=1, keepdims=True)
    b.y[:, 10:13] = rng.normal(size=(n, 3)) * np.where(rng.random(n) < 0.3, 0.05, 1.5)[:, None]
    b.last_distance[:] = np.where(rng.random(n) < 0.1, np.nan, np.linalg.norm(b.y[:, 0:3] - b.cur_wp, axis=1) + rng.normal(size=n) * 0.01)
    limit = qo.MAX_STEPS[oname]
    b.current_step[:] = np.where(rng.random(n) < 0.3, limit + rng.integers(-2, 2, n), rng.integers(0, limit, n))
    if oname == "v2":
        b.final_reached[:] = (b.wp_index >= b.n_wp) & (rng.random(n) < 0.9)
        b.wp_index[:] = np.where(b.final_reached, b.n_wp, np.minimum(b.wp_index, b.n_wp - 1))
        b.cur_wp = b.wp_list[ar, np.minimum(b.wp_index, b.n_wp - 1)].copy()
        b.counter[:] = np.where(b.final_reached, np.where(rng.random(n) < 0.5, 500 + rng.integers(-2, 3, n), rng.integers(0, 500, n)), 0)
        b.final_yaw[:] = rng.uniform(-np.pi, np.pi, n)
    else:
        b.wp_index[:] = np.minimum(b.wp_index, b.n_wp - 1)
        b.cur_wp = b.wp_list[ar, b.wp_index].copy()
    return b


@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
@pytest.mark.parametrize("variant", ["v2", "v1", "v2m"])
def test_randomised_states_dyn_step_matches_dyn_oracle(hh, variant, f32):
    """1,500 random states x random parameters per variant through the device headers' randomised step (the folded form: F/k_m,
    M/k_I, wind acceleration) and the oracle's direct form (true mass, k_I*I, I^-1/k_I): state and reward to 1e-11 (float64 RK4)
    or 1e-4 (float32), flags exact away from the thresholds."""
    rng = np.random.default_rng({"v2": 11, "v1": 12, "v2m": 13}[variant] + 10 * f32)
    oname = "v1" if variant == "v1" else "v2"
    ver = {"v2": 2, "v1": 1, "v2m": 3}[variant]
    n = 1500
    b = _random_batch(rng, variant, n)
    dyn = do.dynamics_draw(int(rng.integers(0, 2**63)), 0.4, 0.4, 0.3, 0.6, np.arange(n), np.zeros(n))
    dyn[: n // 20, 2 + rng.integers(0, 4)] = 0.0                                                   # dead motors
    if f32:
        dyn = dyn.astype(np.float32).astype(np.float64)                                          # what a float32 handle stores
    act = np.stack([rng.uniform(0, 2, n), *rng.uniform(-1, 1, (3, n))], 1).astype(np.float32)
    pre = b.copy()
    with np.errstate(all="ignore"):
        obs_o, rew_o, term_o, trunc_o, info_o = do.step(b, act, substeps=2, **do.dyn_kwargs(dyn))
    tol, tie_eps = (1e-4, 1e-4) if f32 else (1e-11, 1e-12)
    n_flags = 0
    for i in range(n):
        st = dict(y=pre.y[i], wp_list=pre.wp_list[i], n_wp=int(pre.n_wp[i]), wp_index=int(pre.wp_index[i]),
                  last_distance=float(pre.last_distance[i]), current_step=int(pre.current_step[i]), counter=int(pre.counter[i]),
                  final_reached=bool(pre.final_reached[i]), final_yaw=float(pre.final_yaw[i]))
        out, obs, rew, flags, ep_len = hh.step_dyn(ver, st, act[i], dyn[i], f32=f32, substeps=2)
        want = int(term_o[i]) | int(trunc_o[i]) << 1 | (int(info_o[i]) & 0xF) << 2
        dist = np.linalg.norm(b.y[i, 0:3] - pre.cur_wp[i])
        vn, wn = np.linalg.norm(b.y[i, 3:6]), np.linalg.norm(b.y[i, 10:13])
        tie = min(abs(dist - 0.1), abs(dist - 0.5), abs(b.y[i, 2] - 0.1), abs(np.linalg.norm(b.y[i, 0:3]) - 10), abs(vn - 0.1),
                  abs(wn - 0.1)) < tie_eps * 10
        assert flags == want or tie, (i, flags, want)
        n_flags += flags != 0
        if tie:
            continue
        np.testing.assert_allclose(out["y"], b.y[i], rtol=tol, atol=tol)
        np.testing.assert_allclose(rew, rew_o[i], rtol=tol, atol=tol * (100 if f32 else 1))
        np.testing.assert_allclose(obs, obs_o[i], rtol=1e-5 if not f32 else 1e-4, atol=1e-6 if not f32 else 1e-4)
    assert n_flags > n // 10
