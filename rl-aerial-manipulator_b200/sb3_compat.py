"""Stable-Baselines3 file formats and wrapper surface, without importing SB3.

  QuadVecNormalize          stable_baselines3.common.vec_env.VecNormalize for a QuadVecEnv: same constructor arguments,
                            step_wait / reset / normalize_obs / unnormalize_obs / get_original_obs / save / load; the
                            running statistics live on the GPU (vec_normalize.DeviceVecNormalize)
  load_vecnormalize_pkl     read an SB3 `VecNormalize.save()` pickle (e.g. the reference's
                            initial-implementation-v1/vec_normalize.pkl) into a plain dict
  save_vecnormalize_pkl     write a pickle that real SB3 `VecNormalize.load(path, venv)` accepts: same class paths
                            (stable_baselines3.common.vec_env.vec_normalize.VecNormalize, ...running_mean_std.RunningMeanStd,
                            gymnasium.spaces.box.Box) and the same attribute dictionary as the reference's pkl
  save_policy_zip           write an SB3 model zip by replacing `policy.pth` of a template zip (PPO.load-compatible)
  adam_state_to_blobs /     policy.optimizer.pth (torch Adam state_dict over ActorCriticPolicy.parameters()) to and from the
  blobs_to_adam_state       update kernel's Adam moments and step (blob layout of include/quadsim.h)
  save_model_zip /          the whole SB3 model zip (data, policy.pth, policy.optimizer.pth, ...), used by QuadPPO.save / load
  read_model_zip

Reference call sites: initial-implementation-v1/rl_train_vecN.py:11,39 (VecNormalize(...), env.save("vec_normalize.pkl")),
rl_checkpoint_train_vecN.py:22-28,63-64 (VecNormalize.load), runsim_vecN.py:24-26; model zips: v2/rl_train.py:33-35,
v2/runsim_scaledObs.py:15.
"""
from __future__ import annotations

import contextlib
import io
import json
import pickle
import sys
import types
import zipfile

import numpy as np
import torch

from .policy import H1, H2, H3, NACT, pack_params, unpack_params
from .vec_env import LazyInfos, QuadVecEnv
from .vec_normalize import DeviceVecNormalize

_SB3_VN = "stable_baselines3.common.vec_env.vec_normalize"
_SB3_RMS = "stable_baselines3.common.running_mean_std"
_GYM_BOX = "gymnasium.spaces.box"


class _Bag:
    """Attribute bag standing in for an SB3 / gymnasium class while (un)pickling."""

    def __init__(self, *a, **k):
        pass

    def __setstate__(self, st):
        self.__dict__.update(st)


# What a VecNormalize pickle may reference besides SB3 / gymnasium classes (which become attribute bags): numpy's array /
# scalar / dtype reconstructors and a few plain containers.  Anything else (os.system, builtins.eval, ...) is refused: a
# vec_normalize.pkl from a model zoo is untrusted input.
_NUMPY_OK = {"_reconstruct", "ndarray", "dtype", "scalar", "_frombuffer", "float64", "float32", "int64", "int32", "bool_", "uint8"}
_PLAIN_OK = {("collections", "OrderedDict"), ("builtins", "set"), ("builtins", "frozenset"), ("builtins", "slice"),
             ("builtins", "complex"), ("builtins", "bytearray"), ("_codecs", "encode")}


class _TolerantUnpickler(pickle.Unpickler):
    def find_class(self, module, name):
        top = module.split(".")[0]
        if top in ("stable_baselines3", "gymnasium", "gym"):
            return type(name, (_Bag,), {"__module__": module})
        if (top == "numpy" and name in _NUMPY_OK) or (module, name) in _PLAIN_OK:
            return super().find_class(module, name)
        raise pickle.UnpicklingError(f"vec_normalize pickle references {module}.{name}, which is not on the allowlist")


def load_vecnormalize_pkl(path: str) -> dict:
    """obs_rms / ret_rms statistics and hyper-parameters of an SB3 VecNormalize pickle."""
    with open(path, "rb") as f:
        vn = _TolerantUnpickler(f).load()
    d = vn.__dict__
    o, r = d["obs_rms"].__dict__, d["ret_rms"].__dict__
    return {"obs_mean": np.asarray(o["mean"], np.float64), "obs_var": np.asarray(o["var"], np.float64), "obs_count": float(o["count"]),
            "ret_mean": float(r["mean"]), "ret_var": float(r["var"]), "ret_count": float(r["count"]),
            "clip_obs": float(d["clip_obs"]), "clip_reward": float(d["clip_reward"]), "gamma": float(d["gamma"]),
            "epsilon": float(d["epsilon"]), "norm_obs": bool(d["norm_obs"]), "norm_reward": bool(d["norm_reward"]),
            "training": bool(d.get("training", True)), "num_envs": int(d["num_envs"])}


@contextlib.contextmanager
def _spoofed_classes():
    """Classes whose pickled path is SB3's / gymnasium's.  When the real packages are importable they are used as is."""
    made = []

    def get(module, name):
        try:
            mod = __import__(module, fromlist=[name])
            return getattr(mod, name)
        except Exception:  # noqa: BLE001 - package absent: register a stand-in under the same dotted path
            parts = module.split(".")
            for i in range(1, len(parts) + 1):
                mn = ".".join(parts[:i])
                if mn not in sys.modules:
                    sys.modules[mn] = types.ModuleType(mn)
                    made.append(mn)
            cls = type(name, (_Bag,), {"__module__": module, "__qualname__": name})
            setattr(sys.modules[module], name, cls)
            return cls
    try:
        yield get(_SB3_VN, "VecNormalize"), get(_SB3_RMS, "RunningMeanStd"), get(_GYM_BOX, "Box")
    finally:
        for mn in reversed(made):
            sys.modules.pop(mn, None)


def _box_state(low, high, dtype=np.float32) -> dict:
    low, high = np.asarray(low, dtype=dtype), np.asarray(high, dtype=dtype)
    rep = lambda a: str(a.flat[0]) if np.all(a == a.flat[0]) else str(a)   # gymnasium's short repr
    return {"dtype": np.dtype(dtype), "_shape": low.shape, "low": low, "bounded_below": np.isfinite(low) & (low > -np.inf),
            "high": high, "bounded_above": np.isfinite(high) & (high < np.inf), "low_repr": rep(low), "high_repr": rep(high),
            "_np_random": None}


def save_vecnormalize_pkl(path: str, state: dict, num_envs: int, obs_dim: int) -> None:
    """Pickle with SB3's VecNormalize layout (attribute set of the reference's vec_normalize.pkl)."""
    with _spoofed_classes() as (VN, RMS, Box):
        def bag(cls, d):
            o = cls.__new__(cls)
            o.__dict__.update(d)
            return o
        obs_rms = bag(RMS, {"mean": np.asarray(state["obs_mean"], np.float64), "var": np.asarray(state["obs_var"], np.float64),
                            "count": float(state["obs_count"])})
        ret_rms = bag(RMS, {"mean": np.float64(state["ret_mean"]), "var": np.float64(state["ret_var"]), "count": float(state["ret_count"])})
        inf = np.full(obs_dim, np.inf, dtype=np.float32)
        d = {"num_envs": int(num_envs), "observation_space": bag(Box, _box_state(-inf, inf)),
             "action_space": bag(Box, _box_state([0, -1, -1, -1], [2.0, 1, 1, 1])),
             "reset_infos": [{} for _ in range(num_envs)], "_seeds": [None] * num_envs, "_options": [{} for _ in range(num_envs)],
             "render_mode": None, "metadata": {"render_modes": []}, "norm_obs": bool(state.get("norm_obs", True)), "norm_obs_keys": None,
             "obs_rms": obs_rms, "ret_rms": ret_rms, "clip_obs": float(state.get("clip_obs", 10.0)),
             "clip_reward": float(state.get("clip_reward", 10.0)), "gamma": float(state.get("gamma", 0.99)),
             "epsilon": float(state.get("epsilon", 1e-8)), "training": bool(state.get("training", True)),
             "norm_reward": bool(state.get("norm_reward", False)), "old_reward": np.zeros(num_envs), "old_obs": np.zeros((num_envs, obs_dim), np.float32)}
        if not issubclass(VN, _Bag):
            # the real SB3 class: its __getstate__ deletes these three from a copy of __dict__ before pickling
            d.update(venv=None, class_attributes={}, returns=np.zeros(num_envs))
        with open(path, "wb") as f:
            pickle.dump(bag(VN, d), f, protocol=4)


def save_policy_zip(template_zip: str, out_path: str, state_dict: dict) -> None:
    """SB3 model zip = template (data json, optimizer, versions) with `policy.pth` replaced by `state_dict`."""
    buf = io.BytesIO()
    torch.save({k: torch.as_tensor(np.asarray(v)) for k, v in state_dict.items()}, buf)
    with zipfile.ZipFile(template_zip) as zin, zipfile.ZipFile(out_path, "w", zipfile.ZIP_DEFLATED) as zout:
        for item in zin.infolist():
            zout.writestr(item, buf.getvalue() if item.filename == "policy.pth" else zin.read(item.filename))


# ---- policy.optimizer.pth: torch.optim.Adam.state_dict() over ActorCriticPolicy.parameters() ---------------------------------
# parameters() yields the module's own parameter (log_std) first, then the submodules' in registration order; policy.pth's
# state_dict keys come in the same order.
SB3_PARAM_ORDER = ("log_std",) + tuple(f"mlp_extractor.{net}.{i}.{w}" for net in ("policy_net", "value_net") for i in (0, 2, 4)
                                       for w in ("weight", "bias")) + ("action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias")


def pack_params_len(obs_dim: int) -> int:
    """Floats in the parameter blob of include/quadsim.h (qs_policy_param_count), computed on the host."""
    return sum(k_in * k_out + k_out for k_in, k_out in ((obs_dim, H1), (H1, H2), (H2, H3))) * 2 + 2 * (H3 * NACT + NACT) + NACT


def _sb3_shapes(obs_dim: int) -> dict:
    return {k: v.shape for k, v in unpack_params(np.zeros(pack_params_len(obs_dim), np.float32), obs_dim).items()}


def adam_state_to_blobs(opt_state: dict, param_names, obs_dim: int):
    """policy.optimizer.pth (a torch Adam state_dict) -> (m, v) float32 blobs in the layout of include/quadsim.h, the step count
    and the first param_group without its `params`.  param_names: the parameter order (policy.pth's key order).  A state without
    entries (an optimizer that never stepped) gives zero moments and step 0.  Raises ValueError on a parameter count or shape
    that does not match the policy, or unequal per-parameter steps."""
    names = list(param_names)
    shapes = _sb3_shapes(obs_dim)
    if sorted(names) != sorted(shapes):
        raise ValueError(f"policy parameters {names} are not the {len(shapes)} of an SB3 MlpPolicy with {obs_dim} observations")
    ids = [i for g in opt_state["param_groups"] for i in g["params"]]
    if len(ids) != len(names):
        raise ValueError(f"optimizer state covers {len(ids)} parameters, the policy has {len(names)}")
    state = opt_state["state"]
    if not state:
        z = np.zeros(pack_params_len(obs_dim), np.float32)
        return z, z.copy(), 0, {k: v for k, v in opt_state["param_groups"][0].items() if k != "params"}
    m, v, steps = {}, {}, set()
    for pid, name in zip(ids, names):
        if pid not in state:
            raise ValueError(f"optimizer state has no entry for parameter {pid} ({name})")
        s = state[pid]
        for key, out in (("exp_avg", m), ("exp_avg_sq", v)):
            t = np.asarray(torch.as_tensor(s[key]).detach().cpu().float().numpy())
            if t.shape != shapes[name]:
                raise ValueError(f"{key} of {name}: shape {t.shape}, expected {shapes[name]}")
            out[name] = t
        steps.add(float(torch.as_tensor(s["step"]).item()))
    if len(steps) != 1:
        raise ValueError(f"optimizer state has unequal per-parameter steps {sorted(steps)}")
    step = steps.pop()
    if step < 0 or step != int(step):
        raise ValueError(f"optimizer step {step} is not a non-negative integer")
    group = {k: v for k, v in opt_state["param_groups"][0].items() if k != "params"}
    return pack_params(m, obs_dim), pack_params(v, obs_dim), int(step), group


def blobs_to_adam_state(m: np.ndarray, v: np.ndarray, step: int, obs_dim: int, lr: float, betas=(0.9, 0.999), eps: float = 1e-5,
                        param_names=SB3_PARAM_ORDER) -> dict:
    """(m, v, step) of the update kernel -> the state_dict of a real torch.optim.Adam(params, lr, betas, eps) over parameters of
    SB3's shapes in `param_names` order: the installed torch's own format (param_groups, tensor steps)."""
    n = pack_params_len(obs_dim)
    m, v = np.asarray(m, np.float32), np.asarray(v, np.float32)
    if m.shape != (n,) or v.shape != (n,):
        raise ValueError(f"Adam moments must be float32[{n}], got {m.shape} and {v.shape}")
    shapes = _sb3_shapes(obs_dim)
    names = list(param_names)
    if sorted(names) != sorted(shapes):
        raise ValueError(f"param_names {names} are not the {len(shapes)} parameters of an SB3 MlpPolicy")
    params = [torch.nn.Parameter(torch.zeros(shapes[k])) for k in names]
    opt = torch.optim.Adam(params, lr=lr, betas=tuple(betas), eps=eps)
    if int(step) > 0:
        for p in params:
            p.grad = torch.zeros_like(p)
        opt.step()                                   # lets torch create its per-parameter state in its own format
        sm, sv = unpack_params(m, obs_dim), unpack_params(v, obs_dim)
        with torch.no_grad():
            for p, k in zip(params, names):
                st = opt.state[p]
                st["step"].fill_(int(step))
                st["exp_avg"].copy_(torch.from_numpy(sm[k]))
                st["exp_avg_sq"].copy_(torch.from_numpy(sv[k]))
    elif m.any() or v.any():
        raise ValueError("Adam step 0 with nonzero moments")
    return opt.state_dict()


# ---- model zip ------------------------------------------------------------------------------------------------------------
SB3_VERSION = "2.6.0"
# `data` entries SB3 2.6.0 stores as plain JSON (not cloudpickled); clip_range is a pickled schedule in SB3's own zips and a
# float in the ones written here
PLAIN_DATA_FIELDS = ("num_timesteps", "_n_updates", "n_steps", "batch_size", "n_epochs", "gamma", "gae_lambda", "ent_coef", "vf_coef",
                     "max_grad_norm", "learning_rate", "normalize_advantage", "clip_range")
# The exact-resume state (QuadPPO.save).  Not a .pth member: SB3's load_from_zip_file hands every *.pth member to set_parameters,
# which rejects unknown names; other members are ignored.
RESUME_MEMBER = "quadppo_resume.npz"


def _torch_bytes(obj) -> bytes:
    buf = io.BytesIO()
    torch.save(obj, buf)
    return buf.getvalue()


def _system_info() -> str:
    import platform
    return (f"- OS: {platform.platform()} {platform.version()}\n- Python: {platform.python_version()}\n- Stable-Baselines3: {SB3_VERSION}\n"
            f"- PyTorch: {torch.__version__}\n- GPU Enabled: {torch.cuda.is_available()}\n- Numpy: {np.__version__}\n")


def save_model_zip(path: str, state_dict: dict, optimizer_state: dict, data: dict, template_zip: str | None = None,
                   extra: dict | None = None) -> None:
    """Write an SB3 2.6.0 model zip: data, policy.pth, policy.optimizer.pth, pytorch_variables.pth, _stable_baselines3_version,
    system_info.txt, plus the `extra` members {name: bytes} (stored uncompressed).  policy.pth is written in SB3's parameter order
    (SB3_PARAM_ORDER), which is also the order of the optimizer state; state_dict must hold exactly those parameters.

    template_zip: an SB3 zip whose members are kept: of its `data`, only the entries of PLAIN_DATA_FIELDS that are plain JSON there
    (or absent) are replaced -- pickled entries (policy_class, spaces, schedules) stay as they are -- and the two .pth members are
    replaced.  The result is then as PPO.load-compatible as save_policy_zip's output.  Without a template, `data` holds the plain
    fields only; whether SB3's PPO.load accepts such a zip (it reads policy_class and the spaces from `data`) is unverified."""
    members = {}
    if template_zip is not None:
        with zipfile.ZipFile(template_zip) as zin:
            members = {i.filename: zin.read(i.filename) for i in zin.infolist()}
        d = json.loads(members["data"])
        for k, val in data.items():
            if not isinstance(d.get(k), dict):
                d[k] = val
    else:
        d = dict(data)
        members["pytorch_variables.pth"] = _torch_bytes({})
        members["_stable_baselines3_version"] = SB3_VERSION.encode()
        members["system_info.txt"] = _system_info().encode()
    members["data"] = json.dumps(d, indent=4).encode()
    if sorted(state_dict) != sorted(SB3_PARAM_ORDER):
        raise ValueError(f"state_dict keys {sorted(state_dict)} are not the parameters of an SB3 MlpPolicy")
    # SB3's key order (log_std first), whatever the caller's dict order: readers take the optimizer's parameter order from it
    members["policy.pth"] = _torch_bytes({k: torch.as_tensor(np.asarray(state_dict[k])) for k in SB3_PARAM_ORDER})
    members["policy.optimizer.pth"] = _torch_bytes(optimizer_state)
    order = ["data", "policy.pth", "policy.optimizer.pth", "pytorch_variables.pth", "_stable_baselines3_version", "system_info.txt"]
    names = [k for k in order if k in members] + [k for k in members if k not in order]
    with zipfile.ZipFile(path, "w", zipfile.ZIP_DEFLATED) as z:
        for k in names:
            z.writestr(k, members[k])
        for k, b in (extra or {}).items():
            z.writestr(k, b, compress_type=zipfile.ZIP_STORED)


def read_model_zip(path: str) -> dict:
    """An SB3 model zip -> {"data": the JSON dict (pickled entries left as SB3's {":type:", ":serialized:"} dicts),
    "policy": policy.pth as an ordered dict of float32 arrays, "optimizer": the policy.optimizer.pth state_dict or None,
    "members": {name: bytes} of every other member}."""
    with zipfile.ZipFile(path) as z:
        raw = {i.filename: z.read(i.filename) for i in z.infolist()}
    load = lambda b: torch.load(io.BytesIO(b), weights_only=True, map_location="cpu")
    policy = {k: v.detach().float().numpy() for k, v in load(raw.pop("policy.pth")).items()}
    opt = raw.pop("policy.optimizer.pth", None)
    return {"data": json.loads(raw.pop("data")) if "data" in raw else {}, "policy": policy,
            "optimizer": load(opt) if opt is not None else None, "members": raw}


class QuadVecNormalize:
    """SB3 `VecNormalize` semantics over a QuadVecEnv, statistics updated and applied on the device."""

    def __init__(self, venv: QuadVecEnv, training: bool = True, norm_obs: bool = True, norm_reward: bool = True,
                 clip_obs: float = 10.0, clip_reward: float = 10.0, gamma: float = 0.99, epsilon: float = 1e-8):
        self.venv = venv
        self.num_envs, self.observation_space, self.action_space = venv.num_envs, venv.observation_space, venv.action_space
        self._dev = DeviceVecNormalize(venv.sim, norm_obs=norm_obs, norm_reward=norm_reward, clip_obs=clip_obs, clip_reward=clip_reward,
                                       gamma=gamma, epsilon=epsilon, training=training)
        self.old_obs = None
        self.old_reward = None
        n, d = venv.num_envs, venv.sim.obs_dim
        self._h_raw = [torch.empty((n, d), dtype=torch.float32).pin_memory() for _ in range(2)]
        self._h_raw_rew = [torch.empty((n,), dtype=venv.sim.real_dtype).pin_memory() for _ in range(2)]
        venv._transform = self._device_transform

    # properties mirroring SB3's attributes
    training = property(lambda self: self._dev.training, lambda self, v: setattr(self._dev, "training", bool(v)))
    norm_obs = property(lambda self: self._dev.norm_obs)
    norm_reward = property(lambda self: self._dev.norm_reward, lambda self, v: setattr(self._dev, "norm_reward", bool(v)))
    clip_obs = property(lambda self: self._dev.clip_obs)
    gamma = property(lambda self: self._dev.gamma)
    epsilon = property(lambda self: self._dev.epsilon)

    @property
    def obs_rms(self):
        st = self._dev.state_dict()
        return types.SimpleNamespace(mean=st["obs_mean"], var=st["obs_var"], count=st["obs_count"])

    @property
    def ret_rms(self):
        st = self._dev.state_dict()
        return types.SimpleNamespace(mean=st["ret_mean"], var=st["ret_var"], count=st["ret_count"])

    def _device_transform(self, out):
        """Runs on the env's stream right after the step kernel: keep the raw obs/reward for get_original_*, update the
        running statistics (device reduction; NCCL all-gather when sharded), normalise."""
        flip = self.venv._flip
        self._h_raw[flip].copy_(out.obs, non_blocking=True)
        self._h_raw_rew[flip].copy_(out.reward, non_blocking=True)
        dv = self._dev
        if dv.training:
            if dv.norm_obs:
                dv.obs_rms.update(out.obs)
            dv.update_returns(out)
        obs = dv.obs_rms.normalize(out.obs, dv.norm_obs_buf, dv.epsilon, dv.clip_obs) if dv.norm_obs else out.obs
        rew = out.reward
        if dv.norm_reward:
            rew = torch.clamp(rew / torch.sqrt(dv.ret_rms.var[0] + dv.epsilon), -dv.clip_reward, dv.clip_reward).to(out.reward.dtype)
        return obs, rew

    def reset(self):
        raw = self.venv.reset()
        self.old_obs = raw
        self._dev.returns.zero_()
        dev_obs = self.venv.sim.obs
        if self._dev.training and self._dev.norm_obs:
            self._dev.obs_rms.update(dev_obs)
        return self.normalize_obs(raw)

    def step_async(self, actions):
        self.venv.step_async(actions)

    def step_wait(self):
        obs, rewards, dones, infos = self.venv.step_wait()
        flip = self.venv._flip
        self.old_obs, self.old_reward = self._h_raw[flip].numpy(), self._h_raw_rew[flip].numpy()
        if self._dev.norm_obs:   # SB3 normalises info["terminal_observation"] as well
            ids = infos.done_indices if isinstance(infos, LazyInfos) else np.nonzero(dones)[0]
            for i in ids:
                info = infos[int(i)]
                if "terminal_observation" in info:
                    info["terminal_observation"] = self.normalize_obs(info["terminal_observation"])
        return obs, rewards, dones, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def normalize_obs(self, obs: np.ndarray) -> np.ndarray:
        if not self._dev.norm_obs:
            return obs
        st = self._dev.state_dict()
        return np.clip((obs - st["obs_mean"]) / np.sqrt(st["obs_var"] + self._dev.epsilon), -self._dev.clip_obs, self._dev.clip_obs).astype(np.float32)

    def unnormalize_obs(self, obs: np.ndarray) -> np.ndarray:
        if not self._dev.norm_obs:
            return obs
        st = self._dev.state_dict()
        return obs * np.sqrt(st["obs_var"] + self._dev.epsilon) + st["obs_mean"]

    def get_original_obs(self) -> np.ndarray:
        return np.array(self.old_obs)

    def get_original_reward(self) -> np.ndarray:
        return np.array(self.old_reward)

    def save(self, path: str) -> None:
        save_vecnormalize_pkl(path, dict(self._dev.state_dict(), training=self._dev.training), self.num_envs, self.venv.sim.obs_dim)

    @staticmethod
    def load(path: str, venv: QuadVecEnv) -> "QuadVecNormalize":
        st = load_vecnormalize_pkl(path)
        vn = QuadVecNormalize(venv, training=st["training"], norm_obs=st["norm_obs"], norm_reward=st["norm_reward"], clip_obs=st["clip_obs"],
                              clip_reward=st["clip_reward"], gamma=st["gamma"], epsilon=st["epsilon"])
        vn._dev.load_state_dict(st)
        return vn

    def close(self):
        self.venv.close()

    def __getattr__(self, name):   # VecEnvWrapper forwards everything else
        return getattr(self.venv, name)
