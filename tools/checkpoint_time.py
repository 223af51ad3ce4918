"""Cost of QuadPPO checkpoints (QuadPPO.save / load, evaluation.CheckpointCallback) on one GPU.

    python tools/checkpoint_time.py [--out DIR]

1. save and load wall time (host clock; the device is synchronised before the clock starts and save / load synchronise before they
   return) and the zip size, for a v2 float32 QuadPPO with VecNormalize after one training iteration, at 65,536 and 1,048,576 envs;
   three of each, files in a temporary directory.  Also how long deflating the exact-resume member would take and what it would
   save (it is written stored);
2. the time a CheckpointCallback firing after every iteration adds to a learn() iteration: runs with and without it, alternated,
   per-iteration wall time from the log timestamps (train() ends in a host read of its statistics), first iteration dropped.
Prints the device name and power limit with the numbers."""
import argparse
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
import zipfile
import zlib

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rl_aerial_manipulator_b200 import sb3_compat  # noqa: E402
from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv  # noqa: E402
from rl_aerial_manipulator_b200.evaluation import CheckpointCallback  # noqa: E402
from rl_aerial_manipulator_b200.ppo import QuadPPO  # noqa: E402
from rl_aerial_manipulator_b200.vec_normalize import DeviceVecNormalize  # noqa: E402


def _make(n, **hp):
    env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=0)
    vn = DeviceVecNormalize(env)
    return env, vn, QuadPPO(env, vecnorm=vn, seed=0, **hp)


def save_load(n, tmp, hp):
    env, vn, ppo = _make(n, **hp)
    ppo.learn(ppo.n_steps * n)
    path = os.path.join(tmp, f"ckpt_{n}.zip")
    saves, loads = [], []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ppo.save(path)
        saves.append(time.perf_counter() - t0)
    size = os.path.getsize(path)
    with zipfile.ZipFile(path) as z:
        resume = z.read(sb3_compat.RESUME_MEMBER)
    t0 = time.perf_counter()
    deflated = len(zlib.compress(resume, 6))
    t_deflate = time.perf_counter() - t0
    for _ in range(3):
        env2 = BatchedQuadEnv(n, env_version=2, precision="f32", seed=0)
        vn2 = DeviceVecNormalize(env2)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ppo2 = QuadPPO.load(path, env2, vn2, **hp)
        loads.append(time.perf_counter() - t0)
        del ppo2, vn2
        env2.close()
    env.close()
    return saves, loads, size, len(resume), deflated, t_deflate


def callback_cost(n, tmp, hp, iters=4, rounds=2):
    res = {False: [], True: []}
    for _ in range(rounds):
        for with_cb in (False, True):
            env, vn, ppo = _make(n, **hp)
            stamps = []
            cb = CheckpointCallback(ppo.n_steps, os.path.join(tmp, "cb"), save_vecnormalize=True) if with_cb else None
            torch.cuda.synchronize()
            stamps.append(time.perf_counter())
            ppo.learn(iters * ppo.n_steps * n, log=lambda d: stamps.append(time.perf_counter()), callback=cb)
            res[with_cb] += [b - a for a, b in zip(stamps[1:], stamps[2:])]
            env.close()
            shutil.rmtree(os.path.join(tmp, "cb"), ignore_errors=True)
    return statistics.median(res[False]), statistics.median(res[True]), res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to DIR/checkpoint_time.txt")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("checkpoint_time.py needs a CUDA device")
    lines = []
    say = lambda s: (print(s, flush=True), lines.append(s))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    say(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    tmp = tempfile.mkdtemp(prefix="qs_ckpt_")
    fmt = lambda xs: ", ".join(f"{x:.3f}" for x in xs)
    try:
        for n, hp in ((65536, dict(n_steps=64, n_epochs=10)), (1 << 20, dict(n_steps=16, n_epochs=1))):
            saves, loads, size, r, d, td = save_load(n, tmp, hp)
            say(f"v2 f32 + VecNormalize, {n} envs: save {fmt(saves)} s, load {fmt(loads)} s, zip {size / 1e6:.1f} MB "
                f"(resume member {r / 1e6:.1f} MB stored; deflate level 6 would give {d / 1e6:.1f} MB and take {td:.3f} s)")
        for n, hp in ((65536, dict(n_steps=64, n_epochs=10)), (1 << 20, dict(n_steps=16, n_epochs=1))):
            base, cb, allr = callback_cost(n, tmp, hp)
            say(f"learn() iteration, {n} envs, {hp}: median {base:.3f} s without, {cb:.3f} s with a CheckpointCallback every "
                f"iteration: {cb - base:+.3f} s (without {fmt(allr[False])}; with {fmt(allr[True])})")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "checkpoint_time.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
