"""Cost of the on-device evaluate_policy (rl-aerial-manipulator_b200/evaluation.py, csrc/qs_eval.cu) on one GPU.

    python tools/eval_time.py [--out DIR]

1. qs_eval_record alone, replayed from a CUDA graph, at 65,536 and 1,048,576 envs (synthetic flags: 1 done env in 700 per step,
   n_eval_episodes = 10 n so that no env reaches its target and every done row is written);
2. policy forward + env step + qs_eval_record against policy forward + env step, 1,048,576 v2 float32 envs, the shipped v2 policy
   (tensor impl, deterministic), each as a CUDA graph of 32 steps, alternated over 7 rounds;
3. wall time of evaluate_policy for the shipped v2 policy, 4,096 envs, 10,000 episodes (host clock, ends in a device synchronise;
   one warm-up call first).
CUDA events around graph replays; medians.  Prints the device name and power limit with the numbers."""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rl_aerial_manipulator_b200 import _cabi  # noqa: E402
from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv  # noqa: E402
from rl_aerial_manipulator_b200.evaluation import evaluate_policy, first_slot  # noqa: E402
from rl_aerial_manipulator_b200.policy import MlpPolicyKernel  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "policy_v2.npz")


def time_graph(g, reps=20):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g.replay()
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps * 1e3          # us per replay


def record_alone(n, K=200, rounds=7):
    lib = _cabi.load_library()
    E = 10 * n
    gen = torch.Generator(device="cuda").manual_seed(0)
    flags = ((torch.rand((K, n), device="cuda", generator=gen) < 1 / 700).to(torch.uint8)) * 5        # terminated | success
    ret = torch.randn((K, n), device="cuda", generator=gen)
    ln = torch.randint(1, 2000, (K, n), device="cuda", dtype=torch.int32, generator=gen)
    m = int(first_slot(E, n, [n])[0])
    bufs = [torch.zeros(m, dtype=dt, device="cuda") for dt in (torch.float64, torch.int32, torch.uint8, torch.int32)]
    count = torch.zeros(n, dtype=torch.int32, device="cuda")
    state = torch.zeros(_cabi.EVAL_STATE_WORDS, dtype=torch.int32, device="cuda")
    a = _cabi.QsEvalArgs()
    a.n, a.env_id_offset, a.n_global, a.n_eval_episodes, a.return_is_f64 = n, 0, n, E, 0
    a.count, a.state = count.data_ptr(), state.data_ptr()
    a.ret_out, a.len_out, a.flags_out, a.step_out = (b.data_ptr() for b in bufs)
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.qs_eval_begin(C.byref(a), st()) == 0
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for t in range(K):
            a.flags, a.ep_return, a.ep_len = flags[t].data_ptr(), ret[t].data_ptr(), ln[t].data_ptr()
            assert lib.qs_eval_record(C.byref(a), st()) == 0
    out = []
    for _ in range(rounds):
        assert lib.qs_eval_begin(C.byref(a), st()) == 0      # fresh counts: every replay writes its done rows again
        out.append(time_graph(g, reps=1) / K)
    return statistics.median(out), out


def loop_with_and_without_record(n=1 << 20, K=32, rounds=7):
    lib = _cabi.load_library()
    env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=0)
    env.reset()
    pol = MlpPolicyKernel.from_npz(GOLDEN, device="cuda", impl="tensor")
    E = 10 * n
    m = int(first_slot(E, n, [n])[0])
    bufs = [torch.zeros(m, dtype=dt, device="cuda") for dt in (torch.float64, torch.int32, torch.uint8, torch.int32)]
    count = torch.zeros(n, dtype=torch.int32, device="cuda")
    state = torch.zeros(_cabi.EVAL_STATE_WORDS, dtype=torch.int32, device="cuda")
    a = _cabi.QsEvalArgs()
    a.n, a.env_id_offset, a.n_global, a.n_eval_episodes, a.return_is_f64 = n, 0, n, E, 0
    a.flags, a.ep_return, a.ep_len = env.flags.data_ptr(), env.ep_return.data_ptr(), env.ep_len.data_ptr()
    a.count, a.state = count.data_ptr(), state.data_ptr()
    a.ret_out, a.len_out, a.flags_out, a.step_out = (b.data_ptr() for b in bufs)
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.qs_eval_begin(C.byref(a), st()) == 0

    def step(rec):
        pol.forward(env.obs, None)
        env.step(pol.actions_clipped)
        if rec:
            assert lib.qs_eval_record(C.byref(a), st()) == 0
    for rec in (False, True):
        step(rec)
    torch.cuda.synchronize()
    graphs = {}
    for rec in (False, True):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(K):
                step(rec)
        graphs[rec] = g
    res = {False: [], True: []}
    for _ in range(rounds):
        for rec in (False, True):
            res[rec].append(time_graph(graphs[rec], reps=3) / K)
    env.close()
    return statistics.median(res[False]), statistics.median(res[True]), res


def evaluate_wall(n=4096, E=10_000):
    pol = MlpPolicyKernel.from_npz(GOLDEN, device="cuda", impl="tensor")
    env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=0)
    evaluate_policy(pol, env, E)                             # warm-up (module load, first capture)
    torch.cuda.synchronize()
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        res = evaluate_policy(pol, env, E, full=True)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    env.close()
    return times, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to DIR/eval_time.txt")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_time.py needs a CUDA device")
    lines = []
    say = lambda s: (print(s, flush=True), lines.append(s))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    say(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    for n in (65536, 1 << 20):
        med, allr = record_alone(n)
        say(f"qs_eval_record alone, {n} envs, graph of 200 records, 1 done in 700: median {med:.2f} us/record "
            f"(rounds {', '.join(f'{x:.2f}' for x in allr)})")
    base, with_rec, allr = loop_with_and_without_record()
    say(f"policy + step, 1048576 v2 f32 envs: median {base:.1f} us/step (rounds {', '.join(f'{x:.1f}' for x in allr[False])})")
    say(f"policy + step + qs_eval_record:      median {with_rec:.1f} us/step (rounds {', '.join(f'{x:.1f}' for x in allr[True])})")
    say(f"  difference {with_rec - base:+.1f} us/step ({(with_rec / base - 1) * 100:+.2f} %)")
    times, res = evaluate_wall()
    say(f"evaluate_policy, shipped v2 policy, 4096 envs, 10000 episodes: wall {', '.join(f'{t:.3f}' for t in times)} s "
        f"({res.steps} env steps; success {res.success_rate:.4f}, mean length {float(res.ep_length.double().mean()):.1f}, "
        f"mean return {float(res.ep_return.mean()):.1f})")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "eval_time.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
