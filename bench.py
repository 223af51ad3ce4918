"""bench.py -- env-steps/s of the batched WaypointQuadEnv step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload rollout|step] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over the whole env batch.  Workloads (BASELINE.json `configs`):
  rollout  configs[3]/[4]: v2 env, 1,048,576 envs per GPU, float32: VecNormalize statistics (moments reduced inside the step
           kernel) -> MlpPolicy rollout forward on tcgen05 (weights of the reference's
           checkpoints_from_8_6M/ppo_model_2300000_steps.zip; normalise, sample, clip fused) -> env step (physics + reward +
           termination + obs) -> auto-reset.  Default.
  step     configs[2]-style: the env step alone on pre-generated uniform-random actions.
Envs are independent, so N GPUs run N shards with no data-path collective (weak scaling); the only exchange is the
VecNormalize moment triplet (41 doubles per rank and step: one fused all-gather+merge kernel over NVLink peer memory, NCCL
as fallback) and the max-over-ranks of the timing.

Printed JSON (one line, rank 0): the base contract + `roofline` (dominant kernel: the policy forward against the measured
tensor peak; `roofline_other`: the HBM-bound env step), `cpu_baseline` (the CPU oracle port of the reference step on the host
cores), `e2e` (same metric through the SB3-style VecEnv / predict calls with pinned host buffers, copies inside the timed
region), `gpu_launches`, `clocks`.

--dump-outputs DIR: after the K timed steps, the arrays the last timed step handed its caller (env step: obs, reward, flags,
terminal_obs, ep_return, ep_len; rollout: also the policy's actions, actions_clipped, values, log_prob and the VecNormalize
running statistics) go to DIR/<name>.npy as float32 / float64 (integers as float64), rank 0's shard only.  Per-env arrays keep
a fixed, seeded sample of at most 65,536 envs (their indices in env_index.npy).  Seeds, weights and step counts come from the
arguments alone, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_REAL_STDOUT = None


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
ALGO_BYTES = {("v2", "f32"): 269, ("v2", "f64"): 425, ("v1", "f32"): 249}  # SURVEY.md section 8(d)
POLICY_FLOPS = 60032                                                         # actor + critic MACs x 2, v2 (SURVEY.md section 8(d))


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference's own step on the host cores (oracle/_ref, staged by oracle/make_ref.py), else the oracle port
# --------------------------------------------------------------------------------------------------
_CPU = {}
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def reference_staged() -> bool:
    return os.path.exists(os.path.join(REF_DIR, "MANIFEST.json"))


def _cpu_init(n_env, kind):
    """Pool initializer, one per worker process.
    kind "reference": n_env UNMODIFIED `WaypointQuadEnv` objects (initial-implementation-v2/rl_env_scaledObs.py:9) under the
    gymnasium stub, stepped one after the other with reset-on-done -- SB3's DummyVecEnv.step_wait loop; the env's print()s
    go to /dev/null.
    kind "port": one v2 VecOracle (oracle/quad_oracle.py: float64, the same SciPy LSODA call as quadcopter.py:113, auto-reset)."""
    os.environ["OMP_NUM_THREADS"] = "1"
    import numpy as np

    rng = np.random.default_rng(os.getpid())
    _CPU.update(np=np, rng=rng, n=n_env, kind=kind, lo=np.array([0, -1, -1, -1.0]), hi=np.array([2, 1, 1, 1.0]))
    if kind == "reference":
        os.environ["QS_REFERENCE_ROOT"] = REF_DIR
        os.dup2(os.open(os.devnull, os.O_WRONLY), 1)
        sys.stdout = open(os.devnull, "w")
        from oracle import ref_harness

        np.random.seed(os.getpid() & 0x7FFFFFFF)
        envs = [ref_harness.make_env("v2") for _ in range(n_env)]
        for e in envs:
            e.reset()
        _CPU.update(envs=envs)
    else:
        from oracle import quad_oracle as qo

        vec = qo.VecOracle("v2", n_env, lambda ids, eps: rng.random((len(ids), qo.N_UNIFORMS)), integrator="lsoda")
        vec.reset()
        _CPU.update(vec=vec)


def _cpu_chunk(seconds):
    """Step this worker's envs with uniform-random float32 actions for `seconds`; returns (env-steps, elapsed)."""
    np, rng, n = _CPU["np"], _CPU["rng"], _CPU["n"]
    done, t0 = 0, time.perf_counter()
    while True:
        a = (_CPU["lo"] + (_CPU["hi"] - _CPU["lo"]) * rng.random((n, 4))).astype(np.float32)
        with np.errstate(all="ignore"):
            if _CPU["kind"] == "reference":
                for e, act in zip(_CPU["envs"], a):
                    _, _, terminated, truncated, _ = e.step(act)
                    if terminated or truncated:
                        e.reset()
            else:
                _CPU["vec"].step(a)
        done += n
        if time.perf_counter() - t0 >= seconds:
            return done, time.perf_counter() - t0


class CpuArm:
    """The CPU arm, one process per host core (the SubprocVecEnv-style layout)."""

    def __init__(self, n_env: int = 8, procs: int | None = None, kind: str | None = None):
        import multiprocessing as mp

        self.cores = procs or (os.cpu_count() or 1)
        self.n_env = n_env
        self.kind = kind or ("reference" if reference_staged() else "port")
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_cpu_init, initargs=(n_env, self.kind))

    def sample(self, seconds: float):
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_chunk, [seconds] * self.cores, chunksize=1)
        wall = time.perf_counter() - t0
        return sum(r[0] for r in res), wall

    def close(self):
        self.pool.close()
        self.pool.join()

    def describe(self, total, wall, what):
        who = ("the UNMODIFIED reference WaypointQuadEnv.step + reset-on-done (oracle/_ref, staged by oracle/make_ref.py; gymnasium stub)"
               if self.kind == "reference" else "oracle/quad_oracle.py (NumPy port; same SciPy LSODA call as quadcopter.py:113)")
        return (f"{total} env-steps of v2 (float64, scipy odeint/LSODA, auto-reset, uniform-random float32 actions) by {who}, "
                f"{self.cores} processes x {self.n_env} envs, {what} (wall {wall:.1f} s)")


def cpu_baseline(seconds: float = 12.0) -> dict:
    """Reference step on all host cores (kind "reference" when oracle/_ref is staged), the port's number beside it."""
    out = None
    for kind, secs in ((("reference", seconds), ("port", 4.0)) if reference_staged() else (("port", seconds),)):
        arm = CpuArm(kind=kind)
        arm.sample(0.5)
        total, wall = arm.sample(secs)
        arm.close()
        rec = {"value": total / wall, "unit": UNIT, "cores": arm.cores, "kind": kind, "sample": arm.describe(total, wall, f"one {secs:.0f} s sample")}
        if out is None:
            out = rec
        else:
            out["port"] = rec
    return out


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each "step" is one bounded sample on all host cores; the whole K + W run is sized to ~75 s
    per_step = max(0.02, min(10.0, 75.0 / max(1, args.steps + args.warmup)))
    arm = CpuArm()
    for _ in range(args.warmup):
        arm.sample(per_step)
    total, t0 = 0, time.perf_counter()
    for _ in range(args.steps):
        total += arm.sample(per_step)[0]
    wall = time.perf_counter() - t0
    arm.close()
    value = total / wall
    base = {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
            "sample": arm.describe(total, wall, f"{args.steps} samples of {per_step * 1e3:.0f} ms")}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": wall * 1e3 / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args), "envs_per_process": arm.n_env, "integrator": "scipy odeint (LSODA)",
                       "note": ("the unmodified reference env stepped on all host cores" if arm.kind == "reference" else
                                "CPU oracle port of the reference step (oracle/_ref not staged)") + "; each step = one bounded sample on all host cores"},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows: list[list[str]] = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
                power.append(float(r[2]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:  # noqa: BLE001
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak(key: str, fallback: float) -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))[key]), f"measured (MEASURED_PEAKS.json {key})"
        except Exception:  # noqa: BLE001
            pass
    return fallback, "fallback (B200_PROFILING.md)"


def ncu_traffic_table() -> dict:
    """kernel name -> dram bytes (read + write) per launch at 1,048,576 envs, from the committed `ncu --set full` captures of
    exactly these kernels (profiles/roofline_traffic.json names the .csv each number comes from)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            return {k: v for k, v in json.load(open(p)).items() if isinstance(v, (int, float))}
        except Exception:  # noqa: BLE001
            return {}
    return {}


def workload_name(args) -> str:
    n = args.n_envs
    tag = f"{n // (1 << 20)}M" if n % (1 << 20) == 0 else str(n)
    return f"v2_{args.workload}_{tag}_{args.precision}"


DUMP_MAX_ENVS = 1 << 16       # about 15 MB of .npy files for the v2 rollout outputs
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path: str, per_env: dict, whole: dict, n: int) -> None:
    """Write device tensors as DIR/<name>.npy: `per_env` ([n, ...] rows) on a fixed, seeded sample of the envs, `whole` as they are.
    float64 stays float64, every other dtype becomes float32 (floats) or float64 (integers, exact)."""
    import numpy as np
    import torch

    os.makedirs(path, exist_ok=True)
    idx = np.arange(n) if n <= DUMP_MAX_ENVS else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ENVS, replace=False))
    arrays = {"env_index": idx.astype(np.float64)}
    for name, t in per_env.items():
        arrays[name] = t.index_select(0, torch.from_numpy(idx).to(t.device)).cpu().numpy()
    arrays.update({name: t.cpu().numpy() for name, t in whole.items()})
    for name, a in arrays.items():
        arrays[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64 if a.dtype.kind in "iub" else np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte budget")
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def graph_time(fn, steps, unroll, dev, barrier=None):
    """ms per call of `fn`, replayed from a CUDA graph of `unroll` calls (CUDA events on the replay stream, warm replay first)."""
    import torch

    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for i in range(unroll):
            fn(i)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(unroll):
            fn(i)
    g.replay()
    (barrier or (lambda: torch.cuda.synchronize(dev)))()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(1, steps // unroll)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    (barrier or (lambda: torch.cuda.synchronize(dev)))()
    return e0.elapsed_time(e1) / (reps * unroll), g


def step_extra(n, precision, integrator, dev, seed, steps):
    """One extra workload line: the bare env step (configs[2]) on `n` envs, actions regenerated on the device every step."""
    import torch

    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    env = BatchedQuadEnv(n, env_version=2, precision=precision, integrator=integrator, device=dev.index, seed=seed)
    env.reset()
    lo = torch.tensor([0.0, -1, -1, -1], device=dev)
    span = torch.tensor([2.0, 2, 2, 2], device=dev)
    u, a = torch.empty((n, 4), device=dev), torch.empty((n, 4), device=dev)
    many = integrator == "rk4"          # T steps per launch, actions drawn in the kernel (qs_step_many); LSODA: one launch per step
    # small batches: launch, state round trip and the ramp of a 14-warp-per-SM wave are the floor -- 128 steps per launch (a rollout of the
    # reference's n_steps = 2048 is 16 launches; T = 16 / 32 / 64 / 128 measured 4.01 / 3.77 / 3.61 / 3.38 us per step at 65,536 envs);
    # 1M envs: 4 steps keep the [T, n, ...] record at 0.4 GB
    T = int(os.environ.get("QS_BENCH_T", "0")) or (128 if n <= (1 << 18) else 4)
    if many:
        # T steps per launch, state in registers, uniform actions drawn in the kernel (Philox on (seed, global env id, step))
        ms, graph = graph_time(lambda i: env.step_many(T, update_obs=False), max(8, steps // T), 1, dev)
        ms /= T
        launches, actions = 1.0 / T, f"in-kernel Philox uniform over the action box, {T} steps per launch (qs_step_many)"
    else:
        def one(i):
            u.uniform_()
            torch.addcmul(lo, u, span, out=a)
            env.step(a)
        ms, graph = graph_time(one, steps, 4 if integrator == "rk4" else 1, dev)
        launches, actions = 1, "uniform over the action box, regenerated on the device every step (2 torch kernels inside the timed region)"
    del graph
    env.close()
    algo = ALGO_BYTES[("v2", precision)]
    note = ("parity mode: adaptive LSODA, ~35 divergent f-evals per step -- latency-bound, not a throughput mode" if integrator == "lsoda" else
            ("working set fits the 126 MB L2" if n * 185 < 126e6 else "working set exceeds L2"))
    if many:
        # the state record crosses HBM once per T steps: what is left per env-step is the rollout record (obs 80 B + reward + flags)
        rsz = 4 if precision == "f32" else 8
        state = (84 if precision == "f32" else 160) * 2
        algo = 80 + rsz + 1 + state / T
        note = (f"T = {T} steps per launch: {algo:.1f} algorithmic B per env-step (single-step kernel: {ALGO_BYTES[('v2', precision)]} B); the mode is "
                "bound by the RK4 dependency chains at ~14 warps per SM, not by HBM")
    peak, peak_src = measured_peak("hbm_gbs", 6650.0)
    ach = algo * n / (ms / 1e3) / 1e9
    tag = f"{n // (1 << 20)}M" if n % (1 << 20) == 0 else str(n)
    return {"workload": f"v2_step_{tag}_{precision}" + ("_lsoda" if integrator == "lsoda" else ""), "value": n / (ms / 1e3), "unit": UNIT,
            "ms_per_step": ms, "dtype": precision, "integrator": integrator, "actions": actions, "our_launches_per_step": launches,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
                         "algorithmic_bytes_per_env_step": algo, "note": note}}


def run_gpu(args) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist

    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")        # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    n = args.n_envs                     # per GPU: weak scaling, one shard per rank
    env = BatchedQuadEnv(n, env_version=2, precision=args.precision, integrator="rk4", substeps=args.substeps,
                         device=local, env_id_offset=rank * n, seed=args.seed)
    env.reset()
    policy = vn = fused = None
    torch.cuda.manual_seed(args.seed + rank)          # torch's default CUDA generator: its Philox offset advances under graph replay
    lo = torch.tensor([0.0, -1, -1, -1], device=dev)
    span = torch.tensor([2.0, 2, 2, 2], device=dev)
    fused_holder = {}

    def build_parts(mode):
        """name -> callable(i): the launches of one step, by kernel (also the unit of the per-kernel timing)."""
        parts = {}
        if args.workload == "rollout":
            if mode == "fused":
                from rl_aerial_manipulator_b200.rollout import FusedRollout
                # ONE kernel per step: normalise -> tcgen05 policy forward -> in-kernel Philox Gaussian sampling -> clip -> env step ->
                # auto-reset -> moments (+ merge on one GPU)
                fused_holder["f"] = FusedRollout(env, policy, vecnorm=vn, sample="philox", noise_seed=args.seed)
                parts["rollout_kernel<v2,fused>"] = lambda i: fused_holder["f"].step()
                if vn is not None and world > 1:
                    parts["xchg_merge_kernel"] = lambda i: vn.update_from_moments()
            else:
                # two kernels per step: tcgen05 pipeline policy kernel (normalise, forward, in-kernel Philox sampling, clip) + env step
                if vn is not None and world > 1 and not vn.env_merges:
                    parts["xchg_merge_kernel"] = lambda i: vn.update_from_moments()
                parts["rollout_kernel<v2,policy>"] = lambda i: policy.forward_sampled(env.obs, noise_seed=args.seed, env_id_offset=rank * n,
                                                                                     norm_stats=vn.stats if vn is not None else None)
                parts["env_step_kernel<float,v2,rk4,moments>+moments_final"] = lambda i: env.step(policy.actions_clipped)
        else:
            u, a = torch.empty((n, 4), device=dev), torch.empty((n, 4), device=dev)

            def regen(i):
                u.uniform_()
                torch.addcmul(lo, u, span, out=a)
            parts["torch uniform_ + addcmul (actions, fresh every step)"] = regen
            parts[f"env_step_kernel<{'float' if args.precision == 'f32' else 'double'},v2,rk4>"] = lambda i: env.step(a)
        return parts

    if args.workload == "rollout":
        from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
        from rl_aerial_manipulator_b200.vec_normalize import DeviceRunningMeanStd
        policy = MlpPolicyKernel.from_npz(os.path.join(ROOT, "tests", "golden", "policy_v2.npz"), device=dev)
        if args.vecnorm:
            # VecNormalize(norm_obs=True): the step reduces the moments of the obs it returns; on one GPU the kernel that finishes
            # them also merges them into the running statistics, with several ranks one kernel does the all-gather (2D+1 doubles
            # per rank over NVLink peer memory) and the Chan merge (qs_xchg_merge; NCCL all-gather + merge kernel as fallback)
            vn = DeviceRunningMeanStd(env.obs_dim, dev, exchange=args.vecnorm_exchange)
            # (the fused single-kernel rollout reduces its moments in its own last CTA: the exchange stays a separate launch there)
            vn.attach(env, merge=(world == 1 or (vn.exchange == "peer" and args.rollout == "separate" and not args.split_exchange)))
    parts = build_parts(args.rollout)
    fused = fused_holder.get("f")

    def one_step(i):
        for fn in parts.values():
            fn(i)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()                                                # ranks enter the first exchange together
    for i in range(args.warmup):
        one_step(i)
    barrier()
    # CUDA-graph replay of the step loop (4 steps per graph): removes the host launch path (Python -> ctypes -> cudaLaunch)
    unroll = (4 if args.steps % 4 == 0 else 2 if args.steps % 2 == 0 else 1) if args.graph else 0   # exactly K steps are timed
    graph = None
    if unroll:
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for i in range(unroll):
                one_step(i)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(unroll):
                one_step(i)
        graph.replay()
        barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    if graph is not None:
        for _ in range(args.steps // unroll):
            graph.replay()
    else:
        for i in range(args.steps):
            one_step(i)
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = n * world * args.steps / (ms_total / 1e3)
    if fused is not None and fused.status() != 0:
        raise RuntimeError(f"rollout kernel: an internal hand-over timed out (code {fused.status()}); the timed region is invalid")
    if vn is not None and vn.exchange_failed():
        raise RuntimeError("peer-memory moment exchange timed out waiting for a rank; the timed region is invalid")
    if args.dump_outputs and rank == 0:
        # before anything below steps the env again: the buffers still hold the last timed step's results
        per_env = {"obs": env.obs, "reward": env.reward, "flags": env.flags, "terminal_obs": env.terminal_obs,
                   "ep_return": env.ep_return, "ep_len": env.ep_len}
        src = fused if fused is not None else policy
        if src is not None:
            per_env.update(actions=src.actions, actions_clipped=src.actions_clipped, values=src.values, log_prob=src.logp)
        whole = {"obs_rms_count": vn.count.reshape(1), "obs_rms_mean": vn.mean, "obs_rms_var": vn.var} if vn is not None else {}
        dump_outputs(args.dump_outputs, per_env, whole, n)

    # ---- per-kernel durations for the roofline: each component alone, replayed from its own CUDA graph (no host launch gaps), on one
    # rank at a time only where it has no rendezvous.  With one component the step IS the kernel.
    kernel_ms = {}
    ms_step = ms_total / args.steps
    if len(parts) == 1:
        kernel_ms[next(iter(parts))] = ms_step
    else:
        for name, fn in parts.items():
            if name == "xchg_merge_kernel":
                continue                                   # a rendezvous: its cost is the skew between ranks, reported as the remainder
            kernel_ms[name] = graph_time(fn, 100, 4, dev)[0]
        if "xchg_merge_kernel" in parts:
            kernel_ms["xchg_merge_kernel (rendezvous: remainder of the step)"] = max(0.0, ms_step - sum(kernel_ms.values()))
    barrier()
    # ---- the same rollout workload through the OTHER launch structure (one fused kernel vs policy kernel + step kernel), same process
    pre_extras = []
    if args.workload == "rollout" and world == 1 and not args.no_extras:
        other = "separate" if args.rollout == "fused" else "fused"
        oparts = build_parts(other)
        oms, og = graph_time(lambda i: [fn(i) for fn in oparts.values()], 200, 4, dev)
        del og
        pre_extras.append({"workload": workload_name(args), "rollout": other, "value": n / (oms / 1e3), "unit": UNIT, "ms_per_step": oms,
                           "dtype": args.precision, "kernels": list(oparts),
                           "note": "same workload, the other launch structure (default is the faster one)"})

    # ---- end to end through the SB3-style VecEnv call: pinned host actions in, obs/reward/done out --------
    from rl_aerial_manipulator_b200.vec_env import QuadVecEnv
    del graph
    env.close()
    venv = QuadVecEnv(n, env_version=2, precision=args.precision, substeps=args.substeps, device=local, seed=args.seed,
                      env_id_offset=rank * n, info_mode="lazy")
    obs = venv.reset()
    rng = np.random.default_rng(args.seed + rank)
    host_actions = [(np.array([0, -1, -1, -1.0]) + np.array([2, 2, 2, 2.0]) * rng.random((n, 4))).astype(np.float32) for _ in range(2)]
    e2e_steps = max(3, min(args.steps, 30))

    def e2e_step(i):
        nonlocal obs
        if policy is not None:
            a = policy.predict_host(obs, stochastic=True, norm_stats=vn.stats if vn is not None else None)  # obs H2D -> forward -> actions D2H
        else:
            a = host_actions[i & 1]
        obs, rew, dones, infos = venv.step(a)
        return float(rew[0])

    for i in range(3):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = n * world * e2e_steps / e2e_s
    h2d = venv.h2d_bytes_per_step + (n * venv.sim.obs_dim * 4 if policy is not None else 0)
    d2h = venv.d2h_bytes_per_step + (n * 4 * 4 if policy is not None else 0)
    venv.close()

    if rank == 0:
        peak, peak_src = measured_peak("hbm_gbs", 6650.0)
        tpeak, tsrc = measured_peak("bf16_tflops_sustained", 1400.0)
        algo = ALGO_BYTES[("v2", args.precision)]
        traffic = ncu_traffic_table()
        rl = []
        for name, ms in kernel_ms.items():
            if name.startswith("rollout_kernel"):
                # the tcgen05 pipeline kernel: algorithmic FLOPs (one float32 pass of the two MLPs; the split-float16 mode issues 3x that
                # on the tensor pipe) against the measured dense bf16 GEMM rate.  The fused variant also carries the env step's bytes.
                tach = POLICY_FLOPS * n / (ms / 1e3) / 1e12
                r = {"bound": "tensor", "kernel": name, "achieved": tach, "peak": tpeak, "unit": "TFLOP/s", "frac": tach / tpeak,
                     "traffic": traffic.get(name), "peak_source": tsrc, "algorithmic_flops_per_env_step": POLICY_FLOPS, "kernel_ms": ms,
                     "note": "bound by the epilogues' issue slots (512 tanh + hi/lo split per env: a MUFU holds the issue port ~4.75 cycles, "
                             "F2FP 2, FHFMA 1.33 -- profiles/r02/pipe_rates_b200.txt), not by the tensor pipe; the contract's bounds are "
                             "hbm|tensor, so the fraction is quoted against the measured bf16 GEMM rate"}
                if "fused" in name:
                    hb = (algo + 80 + 16 + 4 + 4) * n / (ms / 1e3) / 1e9      # + obs read, sampled actions, value, log-prob written
                    r["hbm_view"] = {"achieved": hb, "peak": peak, "unit": "GB/s", "frac": hb / peak,
                                     "algorithmic_bytes_per_env_step": algo + 104}
                rl.append(r)
            elif name.startswith("env_step_kernel"):
                ach = algo * n / (ms / 1e3) / 1e9
                rl.append({"bound": "hbm", "kernel": name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                           "traffic": traffic.get(name), "peak_source": peak_src, "algorithmic_bytes_per_env_step": algo, "kernel_ms": ms})
            else:
                rl.append({"kernel": name, "kernel_ms": ms})
        rl.sort(key=lambda r: -r["kernel_ms"])
        roofline = next((r for r in rl if "bound" in r), rl[0])
        roofline_other = [r for r in rl if r is not roofline]
        base = None
        extras = []
        if world == 1 and not args.no_extras:
            # the other single-GPU configurations of BASELINE.json (configs[2] and the float64 modes), short runs in the same process
            extras.extend(pre_extras)
            for (en, prec, integ, st) in ((1 << 20, "f32", "rk4", 200), (1 << 20, "f64", "rk4", 100), (65536, "f32", "rk4", 400),
                                         (65536, "f64", "rk4", 400), (65536, "f64", "lsoda", 6)):
                if args.workload == "step" and en == n and prec == args.precision and integ == "rk4":
                    continue
                extras.append(step_extra(en, prec, integ, dev, args.seed, st))
        if world == 1 and not args.no_cpu_baseline:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-baseline-only"], capture_output=True, text=True)
            try:
                base = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception:  # noqa: BLE001
                base = {"error": (r.stderr or r.stdout)[-300:]}
        ours = sum(1 for k in parts if not k.startswith("torch"))
        if args.workload == "rollout" and args.rollout == "separate" and vn is not None:
            ours += 1                                       # moments_final follows the step kernel
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": args.precision, "data": "synthetic",
                "config": {"workload": workload_name(args), "envs_per_gpu": n, "envs_total": n * world, "integrator": f"rk4x{args.substeps}",
                           "vecnormalize": bool(vn is not None), "cuda_graph": bool(unroll),
                           "rollout": (args.rollout if args.workload == "rollout" else None),
                           "actions": ("policy (ppo_model_2300000_steps weights), Gaussian noise drawn every step "
                                       + "inside the kernel (Philox4x32-10 on seed, global env id, step + Box-Muller)"
                                       + ", clipped to the action box") if policy else "uniform-random over the action box, regenerated on the device every step inside the timed region",
                           "l2": "working set per step (state pool + obs + actions) exceeds the 126 MB L2" if n * 185 > 126e6 else "working set fits L2; no flush between steps",
                           "parallelism": f"env-shard x{world}, no data-path collective",
                           "moment_exchange": (vn.exchange + (" (inside the kernel that finishes the step's moments: qs_step_moments_exchange)"
                                                              if world > 1 and vn.env_merges else "")) if vn is not None else "none"},
                "roofline": roofline, "roofline_other": roofline_other,
                "kernels_ms": kernel_ms, "kernels_ms_sum": sum(kernel_ms.values()),
                "extra": extras, "cpu_baseline": base,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world, "steps": e2e_steps,
                        "api": "QuadVecEnv.step(actions: np.ndarray) -> obs, rewards, dones, infos (pinned staging, info_mode=lazy)"},
                "gpu_launches": ours * args.steps, "clocks": clocks}
        emit(line)
    if world > 1:
        # no destroy_process_group(): tearing down a communicator that a captured CUDA graph still references can block;
        # every rank has passed the final all_reduce, so leave without running the destructors
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--split-exchange", action="store_true", help="N > 1: the moment exchange as its own launch (qs_xchg_merge) instead of "
                    "inside the kernel that finishes the step's moments (A/B)")
    ap.add_argument("--workload", default=None, choices=["rollout", "step"])
    ap.add_argument("--n-envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--substeps", type=int, default=1)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--vecnorm", type=int, default=1, help="rollout workload: update VecNormalize statistics every step (NCCL all-gather when N>1)")
    ap.add_argument("--vecnorm-exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="N>1: how ranks exchange the VecNormalize moments (peer = fused all-gather+merge kernel over NVLink peer memory)")
    ap.add_argument("--graph", type=int, default=1, help="replay the step loop from a CUDA graph (4 steps per graph)")
    ap.add_argument("--rollout", default="separate", choices=["fused", "separate"],
                    help="rollout workload: one fused kernel per step (in-kernel Philox noise), or policy kernel + env-step kernel + torch normal_")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra single-GPU workload lines (configs[2], float64, LSODA)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0; per-env arrays on a fixed sample of <= 65,536 envs)")
    args = ap.parse_args()
    if args.workload is None:
        args.workload = "rollout" if os.path.exists(os.path.join(ROOT, "rl-aerial-manipulator_b200", "policy.py")) else "step"
    if args.cpu_baseline_only:
        print(json.dumps(cpu_baseline()), flush=True)
        return
    # rank 0 must print exactly ONE line on stdout: park the real stdout and send everything else (NCCL's version banner,
    # library chatter) to stderr
    global _REAL_STDOUT
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args)
        return
    run_gpu(args)


if __name__ == "__main__":
    main()
