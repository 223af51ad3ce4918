"""MlpPolicyKernel -- the SB3 `MlpPolicy` rollout forward (actor + critic + Gaussian sampling) as one
fused sm_100a kernel call (`qs_policy_forward`, csrc/qs_policy.cu).

Replaces, for a whole env batch on the device (reference root-relative paths):
    PPO("MlpPolicy", env, policy_kwargs=dict(net_arch=[128, 64, 64], activation_fn=torch.nn.Tanh))
        .policy.forward(obs)            initial-implementation-v2/rl_train.py:27-53, v1/rl_train_vecN.py:13-33
    model.predict(obs, deterministic=True)   initial-implementation-v2/runsim_scaledObs.py:54
Weights come from the SB3 zips the reference ships (`policy.pth` state_dict; keys
mlp_extractor.{policy_net,value_net}.{0,2,4}, action_net, value_net, log_std).
"""
from __future__ import annotations

import ctypes as C
import os
import io
import zipfile

import numpy as np
import torch

from ._cabi import load_library

H1, H2, H3, NACT = 128, 64, 64, 4
ACTION_LOW = (0.0, -1.0, -1.0, -1.0)      # rl_env_scaledObs.py:20-24
ACTION_HIGH = (2.0, 1.0, 1.0, 1.0)


def _bind(lib):
    if getattr(lib, "_policy_bound", False):
        return
    vp, f32 = C.c_void_p, C.c_float
    lib.qs_policy_param_count.argtypes = [C.c_int]
    lib.qs_policy_param_count.restype = C.c_int64
    lib.qs_policy_forward.argtypes = [vp, C.c_int, vp, vp, C.c_int64, vp, f32, f32, vp, vp, vp,
                                      C.POINTER(f32 * 4), C.POINTER(f32 * 4), vp, vp, C.c_int, vp]
    lib.qs_policy_forward.restype = C.c_int
    lib.qs_policy_forward_philox.argtypes = [vp, C.c_int, vp, C.c_int64, C.c_uint64, vp, C.c_int64, vp, f32, f32, vp, vp, vp,
                                             C.POINTER(f32 * 4), C.POINTER(f32 * 4), vp, vp, vp]
    lib.qs_policy_forward_philox.restype = C.c_int
    lib.qs_policy_last_error.restype = C.c_char_p
    lib._policy_bound = True


def pack_params(sd: dict, obs_dim: int) -> np.ndarray:
    """SB3 state_dict -> the blob layout of include/quadsim.h (weights input-major, actor then critic, log_std)."""
    g = lambda k: np.asarray(sd[k], dtype=np.float32)
    parts = []
    for net, head in (("policy_net", "action_net"), ("value_net", "value_net")):
        for i, (k_in, k_out) in zip((0, 2, 4), ((obs_dim, H1), (H1, H2), (H2, H3))):
            w, b = g(f"mlp_extractor.{net}.{i}.weight"), g(f"mlp_extractor.{net}.{i}.bias")
            assert w.shape == (k_out, k_in), (net, i, w.shape)
            parts += [w.T.reshape(-1), b]
        wh, bh = g(f"{head}.weight"), g(f"{head}.bias")
        wpad = np.zeros((H3, NACT), dtype=np.float32)
        bpad = np.zeros(NACT, dtype=np.float32)
        wpad[:, : wh.shape[0]] = wh.T
        bpad[: bh.shape[0]] = bh
        parts += [wpad.reshape(-1), bpad]
    parts.append(g("log_std"))
    return np.concatenate(parts).astype(np.float32)


def unpack_params(blob: np.ndarray, obs_dim: int) -> dict:
    """Inverse of pack_params: the blob -> an SB3-named state_dict (float32)."""
    blob = np.asarray(blob, dtype=np.float32)
    sd, o = {}, 0

    def take(n):
        nonlocal o
        v = blob[o:o + n]
        o += n
        return v
    for net, head, n_out in (("policy_net", "action_net", NACT), ("value_net", "value_net", 1)):
        for i, (k_in, k_out) in zip((0, 2, 4), ((obs_dim, H1), (H1, H2), (H2, H3))):
            sd[f"mlp_extractor.{net}.{i}.weight"] = take(k_in * k_out).reshape(k_in, k_out).T.copy()
            sd[f"mlp_extractor.{net}.{i}.bias"] = take(k_out).copy()
        sd[f"{head}.weight"] = take(H3 * NACT).reshape(H3, NACT)[:, :n_out].T.copy()
        sd[f"{head}.bias"] = take(NACT)[:n_out].copy()
    sd["log_std"] = take(NACT).copy()
    assert o == blob.size
    return sd


IMPL = {"auto": 0, "fp32": 1, "tensor": 2, "tensor_fast": 3, "tensor_pipeline": 4}


class MlpPolicyKernel:
    """impl: "fp32" = CUDA-core FFMA kernel (float32 throughout); "tensor" (or its alias "tensor_pipeline") = the
    warp-specialised tcgen05/TMEM pipeline kernel with split-float16 operands (float32-level accuracy); "tensor_fast" =
    the three-chain tcgen05/TMEM kernel, single float16 operands + MUFU.TANH; "auto" = "tensor" for batches >= 16384 envs,
    "fp32" below.  The tensor kernels clamp each (normalised) observation to +-60,000, inside float16's range, before layer 1
    ("fp32" does not); weights whose value times 2 log2(e) overflows float16 (|w| > ~22,700) are outside their supported range."""

    def __init__(self, state_dict: dict, obs_dim: int, device, impl: str = "auto"):
        self.impl = IMPL[impl]
        self.lib = load_library()
        _bind(self.lib)
        self.obs_dim = int(obs_dim)
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.state_dict = {k: np.asarray(v, dtype=np.float32) for k, v in state_dict.items()}
        blob = pack_params(self.state_dict, self.obs_dim)
        assert blob.size == self.lib.qs_policy_param_count(self.obs_dim)
        self.params = torch.from_numpy(blob).to(self.device)
        self._n = 0
        self._lo = (C.c_float * 4)(*ACTION_LOW)
        self._hi = (C.c_float * 4)(*ACTION_HIGH)
        self._host = None

    # ---- constructors ----------------------------------------------------------------------------
    @classmethod
    def from_npz(cls, path: str, device="cuda", impl: str = "auto"):
        z = np.load(path)
        sd = {k[2:]: z[k] for k in z.files if k.startswith("w.")}
        return cls(sd, sd["mlp_extractor.policy_net.0.weight"].shape[1], device, impl)

    @classmethod
    def from_sb3_zip(cls, path: str, device="cuda", impl: str = "auto"):
        """PPO.load(path) for the policy weights only (`policy.pth` inside the SB3 zip)."""
        with zipfile.ZipFile(path) as z:
            sd = torch.load(io.BytesIO(z.read("policy.pth")), weights_only=True, map_location="cpu")
        sd = {k: v.numpy() for k, v in sd.items()}
        return cls(sd, sd["mlp_extractor.policy_net.0.weight"].shape[1], device, impl)

    # ---- forward ---------------------------------------------------------------------------------
    def _ensure(self, n: int) -> None:
        if n != self._n:
            dev = self.device
            self.actions = torch.empty((n, NACT), dtype=torch.float32, device=dev)
            self.actions_clipped = torch.empty((n, NACT), dtype=torch.float32, device=dev)
            self.values = torch.empty((n,), dtype=torch.float32, device=dev)
            self.logp = torch.empty((n,), dtype=torch.float32, device=dev)
            self._n = n

    def forward(self, obs: torch.Tensor, noise: torch.Tensor | None = None, norm_stats: torch.Tensor | None = None,
                norm_eps: float = 1e-8, norm_clip: float = 10.0, obs_norm_out: torch.Tensor | None = None,
                clip_low=None, clip_high=None):
        """obs f32[n,D] (device).  noise f32[n,4] ~ N(0,1) for a stochastic rollout step, None -> the mean action.
        Returns (actions, values, logp); the box-clipped actions SB3 feeds to env.step are in `actions_clipped`."""
        n = obs.shape[0]
        assert obs.dtype == torch.float32 and obs.is_contiguous() and obs.shape[1] == self.obs_dim and obs.device == self.device
        self._ensure(n)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        if noise is not None:
            assert noise.dtype == torch.float32 and noise.is_contiguous() and tuple(noise.shape) == (n, NACT)
        if norm_stats is not None:
            assert norm_stats.dtype == torch.float64 and norm_stats.numel() == 1 + 2 * self.obs_dim
        rc = self.lib.qs_policy_forward(p(self.params), self.obs_dim, p(obs), p(noise), n, p(norm_stats), norm_eps, norm_clip,
                                        p(obs_norm_out), p(self.actions), p(self.actions_clipped), C.byref(self._lo), C.byref(self._hi),
                                        p(self.values), p(self.logp), self.impl,
                                        C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        if rc != 0:
            raise RuntimeError(f"qs_policy_forward failed ({rc}): {self.lib.qs_policy_last_error().decode()}")
        return self.actions, self.values, self.logp

    def forward_sampled(self, obs: torch.Tensor, noise_seed: int = 0, env_id_offset: int = 0, norm_stats: torch.Tensor | None = None,
                        norm_eps: float = 1e-8, norm_clip: float = 10.0, obs_norm_out: torch.Tensor | None = None):
        """forward() with the Gaussian noise drawn inside the kernel (`qs_policy_forward_philox`: Philox on the seed, the GLOBAL env
        id and a device-resident step counter -- fresh noise on every call and every CUDA-graph replay, shard independent).  Runs on
        the tcgen05 pipeline kernel whatever `impl` says.  Returns (actions, values, logp); `actions_clipped` as in forward()."""
        n = obs.shape[0]
        assert obs.dtype == torch.float32 and obs.is_contiguous() and obs.shape[1] == self.obs_dim and obs.device == self.device
        self._ensure(n)
        if getattr(self, "_philox_counter", None) is None:
            self._philox_counter = torch.zeros(2, dtype=torch.int64, device=self.device)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        rc = self.lib.qs_policy_forward_philox(p(self.params), self.obs_dim, p(obs), n, int(noise_seed) & 0xFFFFFFFFFFFFFFFF,
                                               p(self._philox_counter), int(env_id_offset), p(norm_stats), norm_eps, norm_clip, p(obs_norm_out),
                                               p(self.actions), p(self.actions_clipped), C.byref(self._lo), C.byref(self._hi), p(self.values),
                                               p(self.logp), C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        if rc != 0:
            raise RuntimeError(f"qs_policy_forward_philox failed ({rc}): {self.lib.qs_policy_last_error().decode()}")
        return self.actions, self.values, self.logp

    def _forward_range(self, first: int, count: int, obs, noise, norm_stats, stream) -> None:
        """forward() on rows [first, first + count) of already allocated full-size buffers, ordered on `stream`."""
        sl = slice(first, first + count)
        p = lambda t: C.c_void_p(t[sl].data_ptr()) if t is not None else None
        rc = self.lib.qs_policy_forward(C.c_void_p(self.params.data_ptr()), self.obs_dim, p(obs), p(noise), count,
                                        C.c_void_p(norm_stats.data_ptr()) if norm_stats is not None else None, 1e-8, 10.0, None,
                                        p(self.actions), p(self.actions_clipped), C.byref(self._lo), C.byref(self._hi),
                                        p(self.values), p(self.logp), self.impl, C.c_void_p(stream.cuda_stream))
        if rc != 0:
            raise RuntimeError(f"qs_policy_forward failed ({rc}): {self.lib.qs_policy_last_error().decode()}")

    def predict_host(self, obs_np: np.ndarray, stochastic: bool = False, norm_stats=None, pipeline_chunks: int | None = None) -> np.ndarray:
        """model.predict for a host batch: obs H2D (pinned) -> fused forward -> clipped actions D2H.  From 262,144 rows the batch
        goes through in 4 chunks on separate streams (pipeline_chunks), so observations of chunk c+1 are copied up while chunk c
        is evaluated and its actions come down."""
        n = obs_np.shape[0]
        if pipeline_chunks is None:
            pipeline_chunks = int(os.environ.get("QS_PIPELINE_CHUNKS", "4")) if n >= 262144 else 1
        if pipeline_chunks > 1:
            return self._predict_host_chunked(obs_np, stochastic, norm_stats, pipeline_chunks)
        if self._host is None or self._host[0].shape[0] != n:
            self._host = (torch.empty((n, self.obs_dim), dtype=torch.float32).pin_memory(),
                          torch.empty((n, NACT), dtype=torch.float32).pin_memory(),
                          torch.empty((n, self.obs_dim), dtype=torch.float32, device=self.device),
                          torch.Generator(device=self.device).manual_seed(0))
        h_obs, h_act, d_obs, gen = self._host
        src = torch.from_numpy(np.ascontiguousarray(obs_np, dtype=np.float32))
        if not src.is_pinned():            # QuadVecEnv returns views of pinned buffers: no host memcpy then
            h_obs.numpy()[...] = obs_np
            src = h_obs
        d_obs.copy_(src, non_blocking=True)
        noise = torch.randn((n, NACT), device=self.device, generator=gen) if stochastic else None
        self.forward(d_obs, noise, norm_stats=norm_stats)
        h_act.copy_(self.actions_clipped, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return h_act.numpy()

    def _predict_host_chunked(self, obs_np, stochastic, norm_stats, chunks) -> np.ndarray:
        n = obs_np.shape[0]
        if self._host is None or self._host[0].shape[0] != n:
            self._host = (torch.empty((n, self.obs_dim), dtype=torch.float32).pin_memory(),
                          torch.empty((n, NACT), dtype=torch.float32).pin_memory(),
                          torch.empty((n, self.obs_dim), dtype=torch.float32, device=self.device),
                          torch.Generator(device=self.device).manual_seed(0))
        if getattr(self, "_chunk_streams", None) is None or len(self._chunk_streams) != chunks:
            self._chunk_streams = [torch.cuda.Stream(device=self.device) for _ in range(chunks)]
        h_obs, h_act, d_obs, gen = self._host
        src = torch.from_numpy(np.ascontiguousarray(obs_np, dtype=np.float32))
        if not src.is_pinned():
            h_obs.numpy()[...] = obs_np
            src = h_obs
        self._ensure(n)
        cur = torch.cuda.current_stream(self.device)
        noise = torch.randn((n, NACT), device=self.device, generator=gen) if stochastic else None
        ready = torch.cuda.Event()
        ready.record(cur)
        per = ((n + chunks - 1) // chunks + 127) // 128 * 128
        for st, f in zip(self._chunk_streams, range(0, n, per)):
            c = min(per, n - f)
            sl = slice(f, f + c)
            st.wait_event(ready)
            with torch.cuda.stream(st):
                d_obs[sl].copy_(src[sl], non_blocking=True)
                self._forward_range(f, c, d_obs, noise, norm_stats, st)
                h_act[sl].copy_(self.actions_clipped[sl], non_blocking=True)
        for st in self._chunk_streams:
            st.synchronize()
        return h_act.numpy()
