"""Time DDPG populations: one population launch against the same P learners run one after another.

    python tools/populationbench.py [--out profiles/r07_ddpg_population.json] [--reps 3]

Update: P = 1, 16, 74, 148, 256 members at batch 64 and 256, every member's ring full (4096 transitions).  "population" is
one DDPGPopulation.update (mr_ddpg_update_population, one CTA per member); "solo" is P DDPGLearner.update calls issued back
to back on the same stream (at batch 256 the solo learner takes its data-parallel path, as a user's would).

Training: train_population's iteration with N = 1024 envs per member and K = 64 (one collect of 64 env steps, then 64
updates at batch 64) for P = 1, 16, 148, against P solo iterations of train(collect_steps=64), one member after another.
CUDA events split each iteration into collect and update time.

The host time of one call (population update, one solo update) is measured too: a population launch carries the
members' hyper-parameters and keys as a 29.7 KB parameter block whatever the member count.

Timing: CUDA events after a warm-up of every configuration, the best of --reps.  The GPU's name and power limit are read
in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mr_rl_b200 import VecMREnv  # noqa: E402
from mr_rl_b200.ddpg import DDPGPopulation, OUNoise, PopulationReplay, collect, collect_population  # noqa: E402

DEV = "cuda:0"


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def timed(fn, iters, reps):
    """Best of reps: ms per call of fn over iters calls."""
    fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / iters)
    return best


def filled_replay(P, cap):
    rep = PopulationReplay(P, cap, random_seeds=list(range(P)), device=DEV)
    g = torch.Generator(device=DEV).manual_seed(0)
    for t in (rep.s, rep.a, rep.s2):
        t.copy_(torch.randn(t.shape, generator=g, device=DEV) * 50)
    rep.r.copy_(torch.randn(rep.r.shape, generator=g, device=DEV))
    rep.count = cap
    return rep


def bench_update(P, batch, reps):
    pop = DDPGPopulation(P, device=DEV)
    rep = filled_replay(P, 4096)
    members, rings = [pop.member(p) for p in range(P)], [rep.member(p) for p in range(P)]

    def solo():
        for m, rb in zip(members, rings):
            m.update(rb, batch)
    iters = max(2, 2000 // P)
    t_pop = timed(lambda: pop.update(rep, batch), iters, reps)
    t_solo = timed(solo, max(2, iters // 8), reps)
    return {"members": P, "batch": batch, "population_ms": t_pop, "solo_ms": t_solo,
            "population_updates_per_s": P / t_pop * 1e3, "solo_updates_per_s": P / t_solo * 1e3,
            "speedup": t_solo / t_pop,
            "population_host_us_per_call": host_us(lambda: pop.update(rep, batch)),
            "solo_host_us_per_call": host_us(lambda: members[0].update(rings[0], batch))}


def host_us(fn, calls=32):
    """Host time of one call (Python, ctypes and the launch, which for the population carries its 29.7 KB parameter
    block), best of 5 bursts of calls small enough not to fill the launch queue."""
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(5):
        t0 = time.perf_counter()
        for _ in range(calls):
            fn()
        best = min(best, (time.perf_counter() - t0) / calls * 1e6)
        torch.cuda.synchronize()
    return best


def bench_train(P, reps, N=1024, K=64, cap=1 << 16):
    env = VecMREnv(P * N, device=DEV, noise="philox", seed=0, auto_reset=True, reward_mode="shaped")
    env.reset(noise_var=1.0, a0=1.0)
    pop = DDPGPopulation(P, device=DEV)
    noise = OUNoise(P * N, device=DEV)
    rep = PopulationReplay(P, cap, device=DEV)
    solo_envs = [VecMREnv(N, env_base=p * N, device=DEV, noise="philox", seed=0, auto_reset=True, reward_mode="shaped")
                 for p in range(P)]
    for e in solo_envs:
        e.reset(noise_var=1.0, a0=1.0)
    solo_noise = [OUNoise(N, env_base=p * N, device=DEV) for p in range(P)]
    learners, rings = [pop.member(p) for p in range(P)], [rep.member(p) for p in range(P)]

    def pop_iter(ev):
        ev[0].record()
        collect_population(env, pop, noise, rep, K)
        ev[1].record()
        for _ in range(K):
            pop.update(rep, 64)
        ev[2].record()

    def solo_iter(ev):
        ev[0].record()
        for p in range(P):
            collect(solo_envs[p], learners[p], solo_noise[p], rings[p], K)
        ev[1].record()
        for p in range(P):
            for _ in range(K):
                learners[p].update(rings[p], 64)
        ev[2].record()

    out = {"members": P, "envs_per_member": N, "k": K}
    for name, fn in (("population", pop_iter), ("solo", solo_iter)):
        best = None
        for r in range(reps + 1):                      # the first pass warms up (and fills the rings)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            fn(ev)
            torch.cuda.synchronize()
            t = (ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]))
            if r and (best is None or sum(t) < sum(best)):
                best = t
        out[f"{name}_collect_ms"], out[f"{name}_update_ms"] = best
        out[f"{name}_iteration_ms"] = sum(best)
    out["speedup"] = out["solo_iteration_ms"] / out["population_iteration_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--members", type=int, nargs="*", default=[1, 16, 74, 148, 256])
    ap.add_argument("--train-members", type=int, nargs="*", default=[1, 16, 148])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("populationbench needs a CUDA device")
    res = {**gpu_info(), "update": [], "train": []}
    for batch in (64, 256):
        for P in args.members:
            r = bench_update(P, batch, args.reps)
            print(json.dumps(r), flush=True)
            res["update"].append(r)
    for P in args.train_members:
        r = bench_train(P, args.reps)
        print(json.dumps(r), flush=True)
        res["train"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
