"""PopulationPPO without a GPU: the permutation -> shared-buffer row translation, the argument refusals of the Python class, and
the argument checks of the two population entry points of libquadsim (qs_ppo_pop_*, qs_policy_forward_pop)."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from rl_aerial_manipulator_b200 import population
from rl_aerial_manipulator_b200.population import PopulationPPO, flat_rows


@pytest.mark.parametrize("K,n,T", [(1, 8, 5), (4, 8, 16), (3, 5, 7), (16, 1, 3)])
def test_flat_rows_matches_numpy(K, n, T):
    rng = np.random.default_rng(K * 100 + n)
    perms = np.stack([rng.permutation(T * n) for _ in range(K)])
    got = flat_rows(torch.from_numpy(perms), n, K).numpy()
    # agent a's flat row r is (time r // n, its env r % n), i.e. column a*n + r % n of the shared [T, K*n] buffers
    want = np.empty_like(perms)
    for a in range(K):
        for j, r in enumerate(perms[a]):
            t, e = divmod(int(r), n)
            want[a, j] = t * K * n + a * n + e
    np.testing.assert_array_equal(got, want)
    shared = np.arange(T * K * n).reshape(T, K * n)
    for a in range(K):            # the translated rows of agent a pick exactly its own columns of the shared buffer
        own = shared[:, a * n:(a + 1) * n].reshape(-1)
        np.testing.assert_array_equal(shared.reshape(-1)[got[a]], own[perms[a]])


def _env(n_envs=32, obs_dim=17):
    return types.SimpleNamespace(n_envs=n_envs, obs_dim=obs_dim, device=torch.device("cuda", 0))


@pytest.mark.parametrize("kw,msg", [
    (dict(vecnorm=object()), "VecNormalize"),
    (dict(K=3), "not K \\* n"),
    (dict(env=_env(65536 * 2), K=2), "at most 65536"),
    (dict(n_steps=0), "n_steps"),
    (dict(seeds=[0, 1, 2]), "3 seeds"),
    (dict(hyper=dict(ent_coef=[0.01, 0.0])), "ent_coef"),
    (dict(hyper=dict(learning_rate=[1e-4] * 5)), "learning_rate"),
    (dict(hyper=dict(gamma=[0.99] * 4)), "unknown keys"),
    (dict(state_dicts=[None] * 3), "3 state_dicts"),
])
def test_refusals(kw, msg):
    args = dict(env=_env(), K=4, seeds=[0, 1, 2, 3])
    args.update(kw)
    with pytest.raises(ValueError, match=msg):
        PopulationPPO(**args)


def test_refuses_several_ranks(monkeypatch):
    monkeypatch.setattr(population.dist, "is_initialized", lambda: True)
    monkeypatch.setattr(population.dist, "get_world_size", lambda group=None: 2)
    with pytest.raises(ValueError, match="single-rank"):
        PopulationPPO(_env(), 4, [0, 1, 2, 3])


def test_population_symbols_exported():
    from rl_aerial_manipulator_b200 import _cabi
    lib = _cabi.load_library()
    for name in ("qs_ppo_pop_create", "qs_ppo_pop_destroy", "qs_ppo_pop_set_hyper", "qs_ppo_pop_update", "qs_ppo_pop_state",
                 "qs_policy_forward_pop"):
        assert hasattr(lib, name), name


def test_population_entry_points_refuse_bad_arguments():
    """The argument checks return QS_EINVAL with a message before any device memory is touched: aligned dummy pointers suffice."""
    from rl_aerial_manipulator_b200 import _cabi
    lib = _cabi.load_library()
    ok = 1 << 20
    h = C.c_void_p()
    for d, K in ((16, 1), (21, 4), (20, 0), (17, -3), (20, 65536)):
        assert lib.qs_ppo_pop_create(0, d, K, C.byref(h)) == -1, (d, K)
        assert b"obs_dim 17 or 20" in lib.qs_ppo_last_error()
    assert lib.qs_ppo_pop_create(0, 20, 2, None) == -1
    assert lib.qs_ppo_pop_set_hyper(None, None, None) == -1 and b"null argument" in lib.qs_ppo_last_error()
    assert lib.qs_ppo_pop_state(None, None, None, None) == -1 and b"null handle" in lib.qs_ppo_last_error()

    def upd(**kw):
        a = dict(h=None, params=ok, obs=ok, actions=ok, old_logp=ok, adv=ok, ret=ok, idx=ok, idx_stride=128, B=128, stats=ok)
        a.update(kw)
        return lib.qs_ppo_pop_update(*a.values(), None)
    for k in ("params", "obs", "actions", "old_logp", "adv", "ret", "idx"):
        assert upd(**{k: None}) == -1, k
        assert b"null argument" in lib.qs_ppo_last_error()
    assert upd(B=0) == -1 and upd(idx_stride=127) == -1
    for k in ("params", "actions"):
        assert upd(**{k: ok + 4}) == -1, k
        assert b"16-byte aligned" in lib.qs_ppo_last_error()
    assert upd(idx=ok + 4) == -1 and b"8-byte" in lib.qs_ppo_last_error()
    assert upd(stats=ok + 2) == -1 and b"4-byte" in lib.qs_ppo_last_error()
    assert upd() == -1 and b"null handle" in lib.qs_ppo_last_error()

    lib.qs_policy_last_error.restype = C.c_char_p
    lo = (C.c_float * 4)(0, -1, -1, -1)
    hi = (C.c_float * 4)(2, 1, 1, 1)

    def fwd(**kw):
        a = dict(params=ok, d=20, K=4, obs=ok, noise=ok, n=8, act=ok, act_c=ok, lo=C.byref(lo), hi=C.byref(hi), val=ok, lp=ok)
        a.update(kw)
        return lib.qs_policy_forward_pop(*a.values(), None)
    for k in ("params", "obs", "act", "val", "lp"):
        assert fwd(**{k: None}) == -1, k
        assert b"bad argument" in lib.qs_policy_last_error()
    for kw in (dict(d=16), dict(d=21), dict(K=0), dict(K=65536), dict(n=-1)):
        assert fwd(**kw) == -1, kw
        assert b"obs_dim 17 or 20" in lib.qs_policy_last_error()
    for k in ("params", "obs", "noise", "act", "act_c"):
        assert fwd(**{k: ok + 4}) == -1, k
        assert b"16-byte aligned" in lib.qs_policy_last_error()
    assert fwd(n=0) == 0          # nothing to do, nothing launched
