"""SB3 file formats and wrapper surface (rl-aerial-manipulator_b200/sb3_compat.py, gym_env.py)."""
import os
import pickletools
import zipfile

import numpy as np
import pytest
import torch

from oracle import quad_oracle as qo
from oracle import sb3_oracle as so


def test_vecnormalize_pkl_roundtrip_and_class_paths(tmp_path, golden_dir):
    from rl_aerial_manipulator_b200 import sb3_compat as sc
    z = np.load(os.path.join(golden_dir, "vecnorm_v1.npz"))
    state = {k: z[k] for k in z.files}
    p = str(tmp_path / "vec_normalize.pkl")
    sc.save_vecnormalize_pkl(p, state, num_envs=8, obs_dim=17)
    back = sc.load_vecnormalize_pkl(p)
    np.testing.assert_array_equal(back["obs_mean"], z["obs_mean"])
    np.testing.assert_array_equal(back["obs_var"], z["obs_var"])
    assert back["obs_count"] == float(z["obs_count"]) and back["ret_count"] == float(z["ret_count"])
    assert back["clip_obs"] == 10.0 and back["gamma"] == 0.99 and back["epsilon"] == 1e-8 and back["num_envs"] == 8
    # the pickle names exactly the classes SB3's own pickle names (so VecNormalize.load of real SB3 accepts it)
    names = [arg for op, arg, _ in pickletools.genops(open(p, "rb").read()) if op.name == "SHORT_BINUNICODE"]
    for want in ("stable_baselines3.common.vec_env.vec_normalize", "VecNormalize", "stable_baselines3.common.running_mean_std",
                 "RunningMeanStd", "gymnasium.spaces.box", "Box"):
        assert want in names
    for key in ("num_envs", "observation_space", "action_space", "reset_infos", "_seeds", "_options", "render_mode", "metadata", "norm_obs",
                "norm_obs_keys", "obs_rms", "ret_rms", "clip_obs", "clip_reward", "gamma", "epsilon", "training", "norm_reward", "old_reward", "old_obs"):
        assert key in names, key       # attribute set of the reference's vec_normalize.pkl
    import sys
    assert "stable_baselines3" not in sys.modules   # the spoofed module entries are removed again


def test_policy_zip_writer(tmp_path, golden_dir):
    from rl_aerial_manipulator_b200 import sb3_compat as sc
    z = np.load(os.path.join(golden_dir, "policy_v2.npz"))
    sd = {k[2:]: z[k] for k in z.files if k.startswith("w.")}
    template = str(tmp_path / "template.zip")
    with zipfile.ZipFile(template, "w") as zf:      # a minimal SB3-shaped zip
        zf.writestr("data", "{}")
        zf.writestr("policy.pth", b"old")
        zf.writestr("_stable_baselines3_version", "2.6.0")
    out = str(tmp_path / "out.zip")
    sd2 = {k: v + 1 for k, v in sd.items()}
    sc.save_policy_zip(template, out, sd2)
    with zipfile.ZipFile(out) as zf:
        assert zf.read("_stable_baselines3_version") == b"2.6.0" and zf.read("data") == b"{}"
    import io
    with zipfile.ZipFile(out) as zf:
        loaded = torch.load(io.BytesIO(zf.read("policy.pth")), weights_only=True)
    assert set(loaded) == set(sd) and torch.equal(loaded["log_std"], torch.from_numpy(sd["log_std"] + 1))


def test_quadcopter_view_matches_reference_formulas():
    from rl_aerial_manipulator_b200.gym_env import QuadcopterView
    from rl_aerial_manipulator_b200 import QUAD
    rng = np.random.default_rng(0)
    q = QuadcopterView()
    for _ in range(20):
        quat = rng.normal(size=4)
        quat /= np.linalg.norm(quat)
        q.state[0:3] = rng.normal(size=3)
        q.state[6:10] = quat
        R = q.rotation_matrix()
        np.testing.assert_allclose(R @ R.T, np.eye(3), atol=1e-12)
        # axis-angle construction of the reference (quaternion.py:46-77)
        theta = 2 * np.arccos(quat[0])
        v = quat[1:] / np.linalg.norm(quat[1:])
        c, s = np.cos(theta), np.sin(theta)
        K = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
        np.testing.assert_allclose(R, c * np.eye(3) + s * K + (1 - c) * np.outer(v, v), atol=1e-12)
        wf = q.world_frame()
        assert wf.shape == (3, 6)
        np.testing.assert_allclose(wf[:, 4], q.state[0:3], atol=1e-12)                       # origin column
        np.testing.assert_allclose(np.linalg.norm(wf[:, 0] - wf[:, 4]), QUAD.arm_length, atol=1e-12)


@pytest.mark.gpu
def test_single_env_facade_vs_oracle():
    """gymnasium-style single env (LSODA parity mode) against the oracle stepping the same state: 1e-9."""
    from rl_aerial_manipulator_b200.gym_env import WaypointQuadEnv
    env = WaypointQuadEnv(env_version=2, seed=11)
    obs, info = env.reset()
    assert obs.shape == (20,) and obs.dtype == np.float32 and info == {}
    b = qo.EnvBatch.empty("v2", 1, max_wp=3)
    b.y[0] = env.quadcopter.state
    b.wp_list[0, 0] = env.waypoint_list[0]
    b.cur_wp[0] = env.current_waypoint
    b.final_yaw[0] = env.final_yaw
    rng = np.random.default_rng(1)
    for t in range(40):
        a = np.array([rng.uniform(0.8, 1.3), *rng.uniform(-0.1, 0.1, 3)], dtype=np.float32)
        o, r, term, trunc, inf = env.step(a)
        oo, ro, to, tro, io = qo.step(b, a[None])
        np.testing.assert_allclose(env.quadcopter.state, b.y[0], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(r, ro[0], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(o, oo[0], rtol=3e-7, atol=1e-9)
        assert term == bool(to[0]) and trunc == bool(tro[0])
        assert env.current_step == t + 1 and np.array_equal(env.quadcopter.position(), env.quadcopter.state[:3])
    assert abs(float(env.F) - float(np.float32(a[0]) * np.float32(0.18) * np.float32(9.81))) == 0
    env.close()


@pytest.mark.gpu
def test_quad_vecnormalize_wrapper_vs_oracle(tmp_path):
    """SB3-surface VecNormalize over QuadVecEnv (NumPy in/out) vs the SB3 restatement; save()/load() round trip."""
    from rl_aerial_manipulator_b200.sb3_compat import QuadVecNormalize, load_vecnormalize_pkl
    from rl_aerial_manipulator_b200.vec_env import QuadVecEnv
    n = 256
    venv = QuadVecEnv(n, env_version=1, obs_scaled=False, precision="f64", seed=4)
    vn = QuadVecNormalize(venv, norm_obs=True, norm_reward=False)
    ref = so.VecNormalizeOracle(n, 17, gamma=0.99)
    obs = vn.reset()
    np.testing.assert_allclose(obs, ref.reset(vn.get_original_obs()), rtol=3e-5, atol=3e-5)
    rng = np.random.default_rng(0)
    n_done = 0
    for t in range(200):
        a = np.stack([rng.uniform(0, 0.4, n), *rng.uniform(-1, 1, (3, n))], 1).astype(np.float32)
        obs, rew, dones, infos = vn.step(a)
        want = ref.step(vn.get_original_obs(), vn.get_original_reward(), dones)
        np.testing.assert_allclose(obs, want, rtol=3e-5, atol=3e-5)
        np.testing.assert_allclose(rew, vn.get_original_reward().astype(np.float32))       # norm_reward=False
        for i in np.nonzero(dones)[0]:
            n_done += 1
            tob = infos[i]["terminal_observation"]
            assert tob.dtype == np.float32 and np.all(np.abs(tob) <= 10.0) and "episode" in infos[i]
    assert n_done > 50
    p = str(tmp_path / "vn.pkl")
    vn.save(p)
    st = load_vecnormalize_pkl(p)
    np.testing.assert_allclose(st["obs_mean"], ref.obs_rms.mean, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(st["obs_var"], ref.obs_rms.var, rtol=1e-8, atol=1e-12)
    venv2 = QuadVecEnv(n, env_version=1, obs_scaled=False, precision="f64", seed=4)
    vn2 = QuadVecNormalize.load(p, venv2)
    assert vn2.norm_obs and not vn2.norm_reward and vn2.gamma == 0.99
    np.testing.assert_array_equal(vn2.obs_rms.mean, vn.obs_rms.mean)
    vn.close()
    vn2.close()


def test_vecnormalize_pkl_with_a_real_sb3_class_on_the_path(tmp_path, golden_dir, monkeypatch):
    """When stable_baselines3 is importable the writer uses its classes; SB3's VecNormalize.__getstate__ deletes `venv`,
    `class_attributes` and `returns` from the state, so they have to be there (ADVICE r01)."""
    import sys
    import types

    from rl_aerial_manipulator_b200 import sb3_compat as sc

    class VecNormalize:                       # the relevant part of SB3 2.6.0's class
        def __getstate__(self):
            state = self.__dict__.copy()
            del state["venv"]
            del state["class_attributes"]
            del state["returns"]
            return state

        def __setstate__(self, state):
            self.__dict__.update(state)
            self.venv = None

    class RunningMeanStd:
        pass

    for mn in ("stable_baselines3", "stable_baselines3.common", "stable_baselines3.common.vec_env", sc._SB3_VN, sc._SB3_RMS):
        monkeypatch.setitem(sys.modules, mn, types.ModuleType(mn))
    VecNormalize.__module__, RunningMeanStd.__module__ = sc._SB3_VN, sc._SB3_RMS
    VecNormalize.__qualname__, RunningMeanStd.__qualname__ = "VecNormalize", "RunningMeanStd"
    sys.modules[sc._SB3_VN].VecNormalize = VecNormalize
    sys.modules[sc._SB3_RMS].RunningMeanStd = RunningMeanStd
    z = np.load(os.path.join(golden_dir, "vecnorm_v1.npz"))
    p = str(tmp_path / "vn.pkl")
    sc.save_vecnormalize_pkl(p, {k: z[k] for k in z.files}, num_envs=8, obs_dim=17)
    back = sc.load_vecnormalize_pkl(p)
    np.testing.assert_array_equal(back["obs_var"], z["obs_var"])
    names = [arg for op, arg, _ in pickletools.genops(open(p, "rb").read()) if op.name == "SHORT_BINUNICODE"]
    assert "venv" not in names and "returns" not in names          # SB3's own pickles do not carry them either


def test_vecnormalize_pkl_reader_refuses_foreign_globals(tmp_path):
    import pickle

    from rl_aerial_manipulator_b200 import sb3_compat as sc

    class Evil:
        def __reduce__(self):
            import os
            return (os.system, ("true",))
    p = str(tmp_path / "evil.pkl")
    with open(p, "wb") as f:
        pickle.dump({"obs_rms": Evil()}, f)
    with pytest.raises(pickle.UnpicklingError, match="allowlist"):
        sc.load_vecnormalize_pkl(p)
