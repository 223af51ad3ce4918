"""Checkpoint file formats on the host: policy.optimizer.pth <-> the update kernel's Adam blobs, the SB3 model zip, and the
CheckpointCallback schedule.  No GPU."""
import io
import json
import os
import zipfile

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as po
from rl_aerial_manipulator_b200 import sb3_compat as sc
from rl_aerial_manipulator_b200.policy import pack_params
from rl_aerial_manipulator_b200.ppo import init_state_dict

D = 20


def _stepped_adam(seed=0, steps=3, lr=2e-4):
    """A real torch Adam(eps=1e-5) over SB3's ActorCriticPolicy parameters, stepped on random gradients."""
    g = torch.Generator().manual_seed(seed)
    net = po.make_torch_actor_critic(init_state_dict(D, seed), D)
    opt = torch.optim.Adam(net.parameters(), lr=lr, eps=1e-5)
    for _ in range(steps):
        for p in net.parameters():
            p.grad = torch.randn(p.shape, generator=g)
        opt.step()
    return net, opt


def test_parameter_order_is_policy_pth_order():
    net, _ = _stepped_adam(steps=0)
    assert tuple(net.state_dict()) == sc.SB3_PARAM_ORDER
    assert [n for n, _ in net.named_parameters()] == list(sc.SB3_PARAM_ORDER)
    assert sc.pack_params_len(D) == pack_params(init_state_dict(D), D).size


def test_optimizer_round_trip():
    net, opt = _stepped_adam()
    orig = opt.state_dict()
    m, v, step, group = sc.adam_state_to_blobs(orig, list(net.state_dict()), D)
    assert step == 3 and m.dtype == np.float32 and m.size == sc.pack_params_len(D)
    back = sc.blobs_to_adam_state(m, v, step, D, group["lr"], group["betas"], group["eps"])
    assert back.keys() == orig.keys()
    assert back["param_groups"] == orig["param_groups"]              # every field, parameter ids in order
    assert list(back["state"]) == list(orig["state"])
    for i, s in orig["state"].items():
        b = back["state"][i]
        assert b.keys() == s.keys()
        for k in s:
            assert b[k].dtype == s[k].dtype and b[k].shape == s[k].shape and torch.equal(b[k], s[k]), (i, k)
    # the written bytes load back through torch as the same state
    buf = io.BytesIO()
    torch.save(back, buf)
    again = torch.load(io.BytesIO(buf.getvalue()), weights_only=True)
    m2, v2, step2, _ = sc.adam_state_to_blobs(again, sc.SB3_PARAM_ORDER, D)
    assert step2 == step and np.array_equal(m2, m) and np.array_equal(v2, v)


def test_fresh_optimizer_round_trip():
    net, opt = _stepped_adam(steps=0)
    m, v, step, _ = sc.adam_state_to_blobs(opt.state_dict(), sc.SB3_PARAM_ORDER, D)
    assert step == 0 and not m.any() and not v.any()
    assert sc.blobs_to_adam_state(m, v, 0, D, 2e-4) == opt.state_dict()


def test_optimizer_refusals():
    net, opt = _stepped_adam()
    sd = opt.state_dict()
    names = list(net.state_dict())
    bad = {"state": dict(sd["state"]), "param_groups": sd["param_groups"]}
    bad["state"][3] = dict(bad["state"][3], exp_avg=torch.zeros(7))
    with pytest.raises(ValueError, match="shape"):
        sc.adam_state_to_blobs(bad, names, D)
    short = {"state": {i: s for i, s in sd["state"].items() if i < 16},
             "param_groups": [dict(sd["param_groups"][0], params=list(range(16)))]}
    with pytest.raises(ValueError, match="parameters"):
        sc.adam_state_to_blobs(short, names, D)
    uneven = {"state": dict(sd["state"]), "param_groups": sd["param_groups"]}
    uneven["state"][5] = dict(uneven["state"][5], step=torch.tensor(7.0))
    with pytest.raises(ValueError, match="unequal"):
        sc.adam_state_to_blobs(uneven, names, D)
    with pytest.raises(ValueError, match="shape"):                       # the policy of the other env version
        sc.adam_state_to_blobs(sd, names, 17)
    with pytest.raises(ValueError, match="MlpPolicy"):
        sc.adam_state_to_blobs(sd, names[:-1] + ["value_net.extra"], D)
    n = sc.pack_params_len(D)
    with pytest.raises(ValueError, match="float32"):
        sc.blobs_to_adam_state(np.zeros(n - 1, np.float32), np.zeros(n, np.float32), 1, D, 2e-4)


DATA = {"num_timesteps": 123456, "_n_updates": 40, "n_steps": 64, "batch_size": 4096, "n_epochs": 10, "gamma": 0.995, "gae_lambda": 0.9,
        "ent_coef": 0.01, "vf_coef": 0.5, "max_grad_norm": 0.5, "learning_rate": 2e-4, "normalize_advantage": True, "clip_range": 0.2}
MEMBERS = ["data", "policy.pth", "policy.optimizer.pth", "pytorch_variables.pth", "_stable_baselines3_version", "system_info.txt"]


def test_model_zip_layout(tmp_path):
    net, opt = _stepped_adam()
    path = str(tmp_path / "m.zip")
    sd = {k: v.detach().numpy() for k, v in net.state_dict().items()}
    sc.save_model_zip(path, sd, opt.state_dict(), DATA, extra={sc.RESUME_MEMBER: b"resume"})
    assert not sc.RESUME_MEMBER.endswith(".pth")
    with zipfile.ZipFile(path) as z:
        assert z.namelist() == MEMBERS + [sc.RESUME_MEMBER]
        assert json.loads(z.read("data")) == DATA
        assert z.read("_stable_baselines3_version") == b"2.6.0"
        assert torch.load(io.BytesIO(z.read("pytorch_variables.pth")), weights_only=True) == {}
        assert z.getinfo(sc.RESUME_MEMBER).compress_type == zipfile.ZIP_STORED
    r = sc.read_model_zip(path)
    assert list(r["policy"]) == list(sd) and all(np.array_equal(r["policy"][k], sd[k]) for k in sd)
    assert r["data"] == DATA and r["members"][sc.RESUME_MEMBER] == b"resume"
    m, v, step, _ = sc.adam_state_to_blobs(r["optimizer"], list(r["policy"]), D)
    m0, v0, step0, _ = sc.adam_state_to_blobs(opt.state_dict(), list(sd), D)
    assert step == step0 and np.array_equal(m, m0) and np.array_equal(v, v0)


def test_model_zip_from_blob_ordered_state_dict(tmp_path):
    """QuadPPO.save passes unpack_params' dict (log_std last); policy.pth must still come out in SB3's order, the order the
    reader pairs the optimizer state with."""
    from rl_aerial_manipulator_b200.policy import unpack_params
    net, opt = _stepped_adam()
    sd = unpack_params(pack_params({k: v.detach().numpy() for k, v in net.state_dict().items()}, D), D)
    assert list(sd) != list(sc.SB3_PARAM_ORDER)
    m, v, step, _ = sc.adam_state_to_blobs(opt.state_dict(), sc.SB3_PARAM_ORDER, D)
    path = str(tmp_path / "m.zip")
    sc.save_model_zip(path, sd, sc.blobs_to_adam_state(m, v, step, D, 2e-4), DATA)
    r = sc.read_model_zip(path)
    assert list(r["policy"]) == list(sc.SB3_PARAM_ORDER)
    m2, v2, step2, _ = sc.adam_state_to_blobs(r["optimizer"], list(r["policy"]), D)
    assert step2 == step and np.array_equal(m2, m) and np.array_equal(v2, v)
    with pytest.raises(ValueError, match="MlpPolicy"):
        sc.save_model_zip(path, dict(sd, extra=np.zeros(1)), opt.state_dict(), DATA)


def test_model_zip_with_template(tmp_path):
    """A synthetic SB3 zip as template: every member but data and the two .pth is copied byte for byte; of `data`, plain
    entries are updated and pickled ones ({":type:", ":serialized:"}) are left alone."""
    tmpl = str(tmp_path / "tmpl.zip")
    pickled = {":type:": "<class 'function'>", ":serialized:": "gAWVAAAA"}
    tdata = {"policy_class": {":type:": "<class 'abc.ABCMeta'>", ":serialized:": "gAWVMAAA"}, "clip_range": pickled, "lr_schedule": pickled,
             "num_timesteps": 1, "n_steps": 2048, "batch_size": 128, "seed": None, "verbose": 1}
    other = {"pytorch_variables.pth": b"\x80\x02}q\x00.", "_stable_baselines3_version": b"2.6.0", "system_info.txt": b"- OS: template\n",
             "extra_member.bin": bytes(range(256))}
    with zipfile.ZipFile(tmpl, "w") as z:
        z.writestr("data", json.dumps(tdata))
        z.writestr("policy.pth", b"old policy")
        z.writestr("policy.optimizer.pth", b"old optimizer")
        for k, b in other.items():
            z.writestr(k, b)
    net, opt = _stepped_adam()
    out = str(tmp_path / "out.zip")
    sc.save_model_zip(out, {k: v.detach().numpy() for k, v in net.state_dict().items()}, opt.state_dict(), DATA, template_zip=tmpl,
                      extra={sc.RESUME_MEMBER: b"x"})
    with zipfile.ZipFile(out) as z:
        assert set(z.namelist()) == {"data", "policy.pth", "policy.optimizer.pth", sc.RESUME_MEMBER, *other}
        for k, b in other.items():
            assert z.read(k) == b, k
        d = json.loads(z.read("data"))
    assert d["policy_class"] == tdata["policy_class"] and d["clip_range"] == pickled and d["lr_schedule"] == pickled
    assert d["seed"] is None and d["verbose"] == 1
    assert all(d[k] == DATA[k] for k in DATA if k != "clip_range")
    r = sc.read_model_zip(out)
    assert list(r["policy"]) == list(sc.SB3_PARAM_ORDER)


class _FakePPO:
    """What the callbacks read: num_timesteps, env.n_envs, world, vecnorm; save() records the file names it was given."""

    def __init__(self, n_envs, vecnorm=None):
        self.env = type("E", (), {"n_envs": n_envs})()
        self.world, self.vecnorm, self.num_timesteps, self.saved = 1, vecnorm, 0, []

    def save(self, path, template_zip=None, vecnormalize_path=None):
        self.saved.append((os.path.basename(path), vecnormalize_path and os.path.basename(vecnormalize_path), template_zip))


@pytest.mark.parametrize("n_envs, n_steps, freq", [(8, 2048, 5000), (512, 32, 32), (512, 32, 50), (4096, 64, 1)])
def test_checkpoint_callback_schedule_and_names(tmp_path, n_envs, n_steps, freq):
    from rl_aerial_manipulator_b200.evaluation import CheckpointCallback
    ppo = _FakePPO(n_envs, vecnorm=object())
    cb = CheckpointCallback(freq, str(tmp_path / "ckpt"), name_prefix="ppo_model", save_vecnormalize=True, template_zip="t.zip")
    cb.init_callback(ppo)
    assert os.path.isdir(tmp_path / "ckpt")
    want = []
    for it in range(1, 13):
        before = ppo.num_timesteps // n_envs
        ppo.num_timesteps += n_steps * n_envs
        if (ppo.num_timesteps // n_envs) // freq != before // freq:     # the iteration crossed a multiple of freq vec-env steps
            want.append((f"ppo_model_{ppo.num_timesteps}_steps.zip", f"ppo_model_vecnormalize_{ppo.num_timesteps}_steps.pkl", "t.zip"))
        assert cb.after_train(ppo) == {}
    assert ppo.saved == want and len(want) > 0


def test_checkpoint_callback_without_vecnormalize(tmp_path):
    from rl_aerial_manipulator_b200.evaluation import CheckpointCallback
    ppo = _FakePPO(4)
    cb = CheckpointCallback(1, str(tmp_path), save_vecnormalize=True)
    cb.init_callback(ppo)
    ppo.num_timesteps = 8
    cb.after_train(ppo)
    assert ppo.saved == [("rl_model_8_steps.zip", None, None)]
    with pytest.raises(ValueError):
        CheckpointCallback(0, str(tmp_path))
    ppo.world = 2
    with pytest.raises(ValueError, match="single-rank"):
        CheckpointCallback(1, str(tmp_path)).init_callback(ppo)


def test_save_and_load_refuse_several_ranks(tmp_path, monkeypatch):
    from rl_aerial_manipulator_b200 import ppo as ppo_mod
    fake = _FakePPO(4)
    fake.world = 2
    with pytest.raises(ValueError, match="single-rank"):
        ppo_mod.QuadPPO.save(fake, str(tmp_path / "x.zip"))
    monkeypatch.setattr(ppo_mod.dist, "is_initialized", lambda: True)
    monkeypatch.setattr(ppo_mod.dist, "get_world_size", lambda *a: 2)
    with pytest.raises(ValueError, match="single-rank"):
        ppo_mod.QuadPPO.load(str(tmp_path / "x.zip"), env=None)
