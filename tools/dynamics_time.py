"""Cost of dynamics randomisation, and what it does to the shipped policy.

    python tools/dynamics_time.py [--out DIR] [--rounds 7]

Timing: one process, armed and unarmed handles alternated round by round, CUDA events around CUDA-graph replays (20 captured
qs_step calls, or 4 captured qs_step_many launches of T = 128), median over the rounds:
  - qs_step, env v2, 1,048,576 envs, float32 and float64 (state + actions + obs > 126 MB of L2: read from HBM every step);
  - qs_step_many, env v2 float32, 65,536 envs, T = 128, actions drawn in the kernel.
Demonstration: the shipped v2 policy (tests/golden/policy_v2.npz, impl "tensor", deterministic, clipped actions) on 4,096 envs,
first episode per env, every parameter nominal except the mass scale, fixed by set_dynamics at 0.8 / 0.9 / 1.0 / 1.1 / 1.2:
success rate and mean episode length per scale.  Prints, and with --out DIR also writes DIR/dynamics_time.txt.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv  # noqa: E402
from rl_aerial_manipulator_b200.policy import MlpPolicyKernel      # noqa: E402

DR = dict(mass=0.3, inertia=0.3, thrust=0.1, wind=0.3)
LO = torch.tensor([0.0, -1, -1, -1])


def device_info() -> str:
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the numbers still stand with the device name
        q = f"nvidia-smi unavailable ({e})"
    return f"{name}; power limit, max SM clock: {q}"


def graph_of(fn, reps):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    return g


def time_graph(g, per_replay, n_replays=5):
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n_replays):
        g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / (n_replays * per_replay)     # us per step / launch


def step_case(n, precision, armed):
    env = BatchedQuadEnv(n, env_version=2, precision=precision, seed=1, dynamics_randomization=DR if armed else None)
    env.reset()
    act = (LO.cuda() + 2.0 * torch.rand((n, 4), device="cuda")).contiguous()
    reps = 20
    return env, graph_of(lambda: env.step(act), reps), reps


def many_case(n, T, armed):
    env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=1, dynamics_randomization=DR if armed else None)
    env.reset()
    env.step_many(T, action_seed=3, update_obs=False)      # allocates the output buffers outside the capture
    reps = 4
    return env, graph_of(lambda: env.step_many(T, action_seed=3, update_obs=False), reps), reps


def ab(make, rounds, label, unit, log):
    cases = {arm: make(arm) for arm in (False, True)}
    res = {False: [], True: []}
    for r in range(rounds):
        for arm in ((False, True) if r % 2 == 0 else (True, False)):
            _, g, reps = cases[arm]
            res[arm].append(time_graph(g, reps))
    m0, m1 = np.median(res[False]), np.median(res[True])
    log(f"{label}: unarmed {m0:.2f} {unit} (min {min(res[False]):.2f}, max {max(res[False]):.2f}), "
        f"armed {m1:.2f} {unit} (min {min(res[True]):.2f}, max {max(res[True]):.2f}), ratio {m1 / m0:.3f}")
    for arm in cases:
        cases[arm][0].close()
    return m1 / m0


def demo(log, n=4096, steps=2100):
    pol = MlpPolicyKernel.from_npz(os.path.join(ROOT, "tests", "golden", "policy_v2.npz"), device="cuda", impl="tensor")
    log(f"shipped v2 policy, {n} envs (float32, RK4 x 1), first episode per env; only the mass scale differs from nominal")
    for k in (0.8, 0.9, 1.0, 1.1, 1.2):
        env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=0, auto_reset=False,
                             dynamics_randomization=dict(mass=0.0, inertia=0.0, thrust=0.0, wind=0.0))
        obs = env.reset()
        env.set_dynamics(mass_scale=k)
        length = torch.zeros(n, dtype=torch.int32, device="cuda")
        fin = torch.zeros(n, dtype=torch.uint8, device="cuda")
        done = torch.zeros(n, dtype=torch.bool, device="cuda")
        for t in range(steps):
            pol.forward(obs, None)
            out = env.step(pol.actions_clipped)
            obs = out.obs
            newly = out.done & ~done
            length[newly] = t + 1
            fin[newly] = out.flags[newly]
            done |= newly
            if t % 64 == 63 and bool(done.all()):
                break
        f = fin.cpu().numpy()
        success = ((f & 0x04) != 0) & ((f & 0x01) != 0)
        crashed = (f & 0x10) != 0
        L = length.cpu().numpy().astype(np.float64)
        log(f"  mass x {k:.1f}: success {success.mean():.4f}, crashed {crashed.mean():.4f}, all done {bool(done.all())}, "
            f"mean episode length {L[done.cpu().numpy()].mean():.1f} (successful {L[success].mean() if success.any() else float('nan'):.1f})")
        env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for dynamics_time.txt (default: print only)")
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dynamics_time.py measures on the GPU; no CUDA device found")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(device_info())
    log(f"dynamics randomisation ranges of the armed handles: {DR}")
    ab(lambda arm: step_case(1 << 20, "f32", arm), args.rounds, "qs_step v2 f32, 1,048,576 envs", "us/step", log)
    ab(lambda arm: step_case(1 << 20, "f64", arm), args.rounds, "qs_step v2 f64, 1,048,576 envs", "us/step", log)
    ab(lambda arm: many_case(65536, 128, arm), args.rounds, "qs_step_many v2 f32, 65,536 envs, T = 128", "us/launch", log)
    demo(log)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "dynamics_time.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
