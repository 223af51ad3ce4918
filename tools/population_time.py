"""Seconds per PPO iteration of K agents at the reference's v1 settings (8 envs per agent, 2,048 steps, batch 128, 10 epochs):
PopulationPPO (all K agents in the same launches) against K solo QuadPPO iterations run back to back (policy_impl="fp32", as
the population's agents).  One warm-up iteration per variant (graph capture), then `--rounds` timed rounds in which the two
variants alternate; a host clock around each variant's work, which ends in a device synchronise.  Prints the card and its power
limit first.
    python tools/population_time.py [--ks 1,4,16,64] [--rounds 3]"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.getcwd())
import torch

from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
from rl_aerial_manipulator_b200.population import PopulationPPO
from rl_aerial_manipulator_b200.ppo import QuadPPO

ap = argparse.ArgumentParser()
ap.add_argument("--ks", default="1,4,16,64")
ap.add_argument("--rounds", type=int, default=3)
args = ap.parse_args()
N_ENVS, T, BS, EPOCHS = 8, 2048, 128, 10
cfg = dict(n_steps=T, batch_size=BS, n_epochs=EPOCHS, gamma=0.995, gae_lambda=0.9)

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
print(f"# {torch.cuda.get_device_name(0)} | nvidia-smi: {smi.stdout.strip()}")
print(f"# v1, {N_ENVS} envs per agent, n_steps {T}, batch {BS}, {EPOCHS} epochs; seconds per iteration (collect + train) of all K agents")


def iteration(ppo):
    ppo.collect_rollouts()
    ppo.train()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


print(f"{'K':>4} {'population s/it':>16} {'K solo s/it':>12} {'speed-up':>9}   (per round: population | solo)")
for K in (int(k) for k in args.ks.split(",")):
    pop = PopulationPPO(BatchedQuadEnv(K * N_ENVS, env_version=1, seed=0), K, list(range(K)), **cfg)
    solos = [QuadPPO(BatchedQuadEnv(N_ENVS, env_version=1, seed=0, env_id_offset=a * N_ENVS), policy_impl="fp32", seed=a, **cfg)
             for a in range(K)]
    timed(lambda: iteration(pop))                     # warm-up: first collection captures the step graph
    timed(lambda: [iteration(s) for s in solos])
    tp, ts = [], []
    for _ in range(args.rounds):
        tp.append(timed(lambda: iteration(pop)))
        ts.append(timed(lambda: [iteration(s) for s in solos]))
    p, s = min(tp), min(ts)
    rounds = " ".join(f"{a:.3f}|{b:.3f}" for a, b in zip(tp, ts))
    print(f"{K:>4} {p:>16.3f} {s:>12.3f} {s / p:>8.2f}x   {rounds}", flush=True)
    pop.close()
    pop.env.close()
    for q in solos:
        q.opt.close()
        q.env.close()
    del pop, solos
    torch.cuda.empty_cache()
