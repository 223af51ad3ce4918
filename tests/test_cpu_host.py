"""CPU-side tests (no GPU): the C-ABI library loads and exports every symbol include/quadsim.h declares, the product
fails loudly without a CUDA device, and the host logic (parameter packing, moment merging across ranks over gloo,
info dictionaries) is correct."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest
import torch

import rl_aerial_manipulator_b200 as qsim
from oracle import sb3_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from rl_aerial_manipulator_b200 import _build
    _build.build(verbose=False)
    return qsim.load_library()


def test_library_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "quadsim.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = sorted(set(re.findall(r"\b(qs_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 18, names
    for n in names:
        assert hasattr(lib, n), f"libquadsim.so does not export {n}"
    assert lib.qs_abi_version() == 3


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure path")
def test_no_cpu_fallback(lib):
    cfg = qsim.make_config(n_envs=4)
    h = C.c_void_p()
    rc = lib.qs_create(C.byref(cfg), C.byref(h))
    assert rc != 0 and not h
    assert b"no CUDA device" in lib.qs_last_error(None) or b"CUDA" in lib.qs_last_error(None)
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        BatchedQuadEnv(4)


def test_config_constants_match_reference_values():
    c = qsim.make_config()
    assert c.mass == 0.18 and c.g == 9.81 and c.dt == 1 / 200
    assert c.max_prop_thrust == 2 * 0.18 * 9.81 / 4 and c.min_prop_thrust == 0.0
    np.testing.assert_allclose(np.array(c.inv_inertia[:]).reshape(3, 3) @ np.array(c.inertia[:]).reshape(3, 3), np.eye(3), atol=1e-12)
    np.testing.assert_allclose(np.array(c.inv_mix[:]).reshape(4, 4) @ np.array(c.mix[:]).reshape(4, 4), np.eye(4), atol=1e-12)
    assert c.sin_tab[0] == np.sin(2 * np.pi) and c.cos_tab[0] == 1.0 and c.lsoda_rtol == 1.49012e-8
    assert c.sin_tab[1] == np.sin(2 * 0.5 * np.pi) and c.sin_tab[3] == np.sin(2 * (1 / 3) * np.pi) and c.cos_tab[4] == np.cos((2 / 3) * (2 * np.pi * 1))
    # values quoted in SURVEY.md section 8(a)
    assert abs(c.inv_inertia[0] - 4000.278) < 1e-3 and abs(c.inv_inertia[8] - 2675.414) < 1e-3 and abs(c.mix[12] - 0.0245499) < 1e-7


def test_policy_param_packing(golden_dir):
    from rl_aerial_manipulator_b200.policy import pack_params, H1, H2, H3, NACT
    z = np.load(os.path.join(golden_dir, "policy_v2.npz"))
    sd = {k[2:]: z[k] for k in z.files if k.startswith("w.")}
    blob = pack_params(sd, 20)
    per = 20 * H1 + H1 + H1 * H2 + H2 + H2 * H3 + H3 + H3 * NACT + NACT
    assert blob.size == 2 * per + NACT

    def run(net_off, x):   # the kernel's arithmetic, in numpy, straight from the blob
        o = net_off
        for k_in, k_out in ((20, H1), (H1, H2), (H2, H3)):
            W = blob[o:o + k_in * k_out].reshape(k_in, k_out); o += k_in * k_out
            b = blob[o:o + k_out]; o += k_out
            x = np.tanh(x @ W + b)
        Wh = blob[o:o + H3 * NACT].reshape(H3, NACT); o += H3 * NACT
        return x @ Wh + blob[o:o + NACT]
    obs = z["obs"].astype(np.float64)
    _, value, _, mean = so.mlp_policy_forward(sd, obs)
    np.testing.assert_allclose(run(0, obs), mean, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(run(per, obs)[:, 0], value, rtol=1e-6, atol=1e-5)
    np.testing.assert_array_equal(blob[-4:], sd["log_std"])
    # the oracle itself reproduces the torch forward recorded from the shipped zip
    np.testing.assert_allclose(mean, z["mean_f64"], rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(value, z["value_f64"], rtol=1e-10, atol=1e-11)


def _np_moments(x):
    x = x.astype(np.float64)
    return np.concatenate([[x.shape[0]], x.mean(0), x.var(0) * x.shape[0]])


def test_merge_of_shards_equals_one_shot():
    from oracle.sb3_oracle import merge_moments
    rng = np.random.default_rng(0)
    x = (rng.normal(size=(4000, 20)) * 3 + 2).astype(np.float32)
    ref = so.RunningMeanStd((20,))
    ref.update(x)
    stats0 = torch.cat([torch.tensor([1e-4], dtype=torch.float64), torch.zeros(20, dtype=torch.float64), torch.ones(20, dtype=torch.float64)])
    for k in (1, 2, 8):
        shards = np.array_split(x, k)
        m = torch.from_numpy(np.stack([_np_moments(s) for s in shards]))
        s = merge_moments(stats0, m).numpy()
        assert abs(s[0] - ref.count) < 1e-9
        np.testing.assert_allclose(s[1:21], ref.mean, rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(s[21:], ref.var, rtol=1e-11, atol=1e-13)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from oracle.sb3_oracle import merge_moments
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    rng = np.random.default_rng(42)
    x = (rng.normal(size=(1024, 17)) * 2 - 1).astype(np.float32)           # the global batch, same on every rank
    stats = torch.cat([torch.tensor([1e-4], dtype=torch.float64), torch.zeros(17, dtype=torch.float64), torch.ones(17, dtype=torch.float64)])
    for step in range(3):
        xs = x[rank::world] * (step + 1)                                        # this rank's shard of envs
        mine = torch.from_numpy(_np_moments(xs))
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)                                         # what DeviceRunningMeanStd.update does over NCCL
        stats = merge_moments(stats, torch.stack(gathered))
    q.put((rank, stats.numpy()))
    dist.destroy_process_group()


def test_vecnormalize_statistics_world_size_2_gloo():
    """N>1 path on CPU: two ranks, each with half the envs, all-gather their moment triplets and end up with the
    statistics SB3's RunningMeanStd computes on the whole batch."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 1000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    np.testing.assert_array_equal(res[0], res[1])                               # ranks agree bit for bit
    rng = np.random.default_rng(42)
    x = (rng.normal(size=(1024, 17)) * 2 - 1).astype(np.float32)
    ref = so.RunningMeanStd((17,))
    for step in range(3):
        ref.update(x * (step + 1))
    assert abs(res[0][0] - ref.count) < 1e-9
    np.testing.assert_allclose(res[0][1:18], ref.mean, rtol=1e-11, atol=1e-12)
    np.testing.assert_allclose(res[0][18:], ref.var, rtol=1e-10, atol=1e-12)


def test_info_dicts_follow_reference_and_sb3_conventions():
    from rl_aerial_manipulator_b200 import _cabi
    from rl_aerial_manipulator_b200.vec_env import QuadVecEnv, LazyInfos

    class Fake:
        monitor = True
        _make_info = QuadVecEnv._make_info

        def _fetch_done(self, ids):
            return np.arange(len(ids) * 20, dtype=np.float32).reshape(len(ids), 20), np.array([12.3456789] * len(ids)), np.array([77] * len(ids)), 1.5
    fk = Fake()
    F = _cabi
    flags = np.array([0, F.FLAG_SUCCESS | F.FLAG_STOPPED, F.FLAG_TERMINATED | F.FLAG_CRASHED, F.FLAG_TRUNCATED,
                      F.FLAG_TERMINATED | F.FLAG_TRUNCATED | F.FLAG_OOB, F.FLAG_TERMINATED | F.FLAG_SUCCESS], dtype=np.uint8)
    dones = (flags & 3) != 0
    infos = LazyInfos(fk, flags, dones)
    assert len(infos) == 6 and infos[0] == {}
    assert infos[1] == {"success": True, "stopped": True}                       # v2 hold phase / first arrival, not done
    assert infos[2]["crashed"] is True and infos[2]["success"] is False and infos[2]["TimeLimit.truncated"] is False
    assert infos[3]["TimeLimit.truncated"] is True and "success" not in infos[3]
    assert infos[4]["out_of_bounds"] is True and infos[4]["TimeLimit.truncated"] is False   # truncated AND terminated -> False
    assert infos[5] == {"success": True, "stopped": False, "TimeLimit.truncated": False,
                        "terminal_observation": infos[5]["terminal_observation"], "episode": {"r": 12.345679, "l": 77, "t": 1.5}}
    np.testing.assert_array_equal(infos.done_indices, [2, 3, 4, 5])
    np.testing.assert_array_equal(infos[3]["terminal_observation"], np.arange(20, 40, dtype=np.float32))


def test_ctypes_structs_match_the_header_layout(tmp_path):
    """The binding's ctypes structures against include/quadsim.h as a C compiler lays them out (gcc, plain C: the header is the ABI
    a maintainer of the reference binds): same size, same offset for every field."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    from rl_aerial_manipulator_b200 import _cabi
    structs = {"qs_config": _cabi.QsConfig, "qs_state_view": _cabi.QsStateView, "qs_rollout_args": _cabi.QsRolloutArgs,
               "qs_step_many_args": _cabi.QsStepManyArgs, "qs_ppo_hyper": _cabi.QsPpoHyper, "qs_pid_gains": _cabi.QsPidGains}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "quadsim.h"', "int main(void) {"]
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True).stdout
    seen = 0
    for ln in out.splitlines():
        cname, field, val = ln.split()
        cls = structs[cname]
        want = C.sizeof(cls) if field == "size" else getattr(cls, field).offset
        assert int(val) == want, (cname, field, int(val), want)
        seen += 1
    assert seen == sum(len(c._fields_) + 1 for c in structs.values())


def test_bench_dump_outputs_sample_and_dtypes(tmp_path):
    """bench.py --dump-outputs: per-env rows on the same seeded env sample every time, float32 / float64 only, within 64 MB."""
    import bench
    n = bench.DUMP_MAX_ENVS + 1000
    g = torch.Generator().manual_seed(0)
    per_env = {"obs": torch.randn((n, 20), generator=g), "reward": torch.randn(n, generator=g, dtype=torch.float64),
               "flags": torch.randint(0, 256, (n,), generator=g, dtype=torch.uint8), "ep_len": torch.arange(n, dtype=torch.int32)}
    whole = {"obs_rms_mean": torch.randn(20, generator=g, dtype=torch.float64)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), per_env, whole, n)
    got = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(got) == ["env_index.npy", "ep_len.npy", "flags.npy", "obs.npy", "obs_rms_mean.npy", "reward.npy"]
    assert all(np.array_equal(a, np.load(tmp_path / "b" / f)) for f, a in got.items())
    idx = got["env_index.npy"].astype(np.int64)
    assert len(idx) == bench.DUMP_MAX_ENVS and np.all(np.diff(idx) > 0) and idx[-1] < n
    assert got["obs.npy"].dtype == np.float32 and np.array_equal(got["obs.npy"], per_env["obs"].numpy()[idx])
    assert got["reward.npy"].dtype == np.float64 and np.array_equal(got["reward.npy"], per_env["reward"].numpy()[idx])
    assert got["flags.npy"].dtype == np.float64 and np.array_equal(got["flags.npy"], per_env["flags"].numpy()[idx])
    assert np.array_equal(got["ep_len.npy"], idx.astype(np.float64))
    assert np.array_equal(got["obs_rms_mean.npy"], whole["obs_rms_mean"].numpy())
    with pytest.raises(RuntimeError, match="budget"):
        bench.dump_outputs(str(tmp_path / "c"), {"obs": torch.zeros((n, 300))}, {}, n)
