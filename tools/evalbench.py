"""Time the greedy evaluation of DDPG populations (evaluate_population) and one round of population-based training.

    python tools/evalbench.py [--out profiles/r08_ddpg_eval.json] [--reps 5]

Evaluation: P = 1, 16, 148 members x N = 128, 1024 episodes each, on the default task (start positions sampled from
init_space, max_timesteps = 50, so K = 51 steps, shaped reward, Philox noise with noise_var = 1, fp64 storage), with the
members' freshly initialised actors (their episodes time out: every env takes all 51 steps).  "population" is one
evaluate_population launch; "solo" is P fused actor rollouts (VecMREnv.rollout with the member's actor, N envs, 51
steps) issued back to back, what a user without the population evaluation would run.  Both on the default 3xFP16 path.

Early exit: P = 148, N = 1024 with the sampled starts against starts inside the goal radius (every episode ends after one
step, so every tile leaves the step loop after one step).

PBT round: P = 148 members, 1024 training envs and 1024 evaluation episodes per member: train (train_population of one
collect launch of 64 steps and 64 population updates at batch 64), evaluate (evaluate_population, with the copy of the
scores to the host), exploit (pbt_plan, DDPGPopulation.exploit and the hyper-parameter perturbation).

Timing: CUDA events after a warm-up of every configuration, the best of --reps.  The GPU's name and power limit are read
in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mr_rl_b200 import VecMREnv  # noqa: E402
from mr_rl_b200.ddpg import (DDPGPopulation, OUNoise, PopulationReplay, evaluate_population, pbt_plan,  # noqa: E402
                             train_population)

DEV = "cuda:0"


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def timed(fn, iters, reps):
    """Best of reps: ms per call of fn over iters calls (after one warm-up call)."""
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


def task_env(n, **kw):
    env = VecMREnv(n, device=DEV, noise="philox", seed=1, reward_mode="shaped", **kw)
    env.reset(noise_var=1.0, a0=1.0)
    return env


def bench_eval(P, N, reps):
    pop = DDPGPopulation(P, seeds=list(range(P)), device=DEV)
    env = task_env(128)
    K = env.max_timesteps + 1
    res = evaluate_population(env, pop, N)
    t_pop = timed(lambda: evaluate_population(env, pop, N), 5, reps)
    solos = [task_env(N) for _ in range(P)]

    def solo():
        for p, e in enumerate(solos):
            e.rollout(policy=pop.actor[p], k_steps=K, accumulate_stats=False)
    t_solo = timed(solo, 2, reps)
    return {"members": P, "member_envs": N, "k_steps": K, "population_ms": t_pop, "solo_ms": t_solo,
            "speedup": t_solo / t_pop, "mean_length": float(res.mean_length.mean()),
            "population_env_steps_per_s": float(res.env_steps.sum()) / t_pop * 1e3}


def bench_early_exit(reps):
    P, N = 148, 1024
    pop = DDPGPopulation(P, seeds=list(range(P)), device=DEV)
    env = task_env(128)
    out = {"members": P, "member_envs": N}
    for name, init in (("init_space", None), ("inside_goal", torch.tensor([10.0, 10.0], dtype=torch.float64))):
        res = evaluate_population(env, pop, N, init=init)
        out[name] = {"ms": timed(lambda: evaluate_population(env, pop, N, init=init), 5, reps),
                     "mean_length": float(res.mean_length.mean())}
    out["ratio"] = out["init_space"]["ms"] / out["inside_goal"]["ms"]
    return out


def bench_pbt_round(reps):
    P, N = 148, 1024
    env = task_env(P * N, auto_reset=True)
    pop = DDPGPopulation(P, seeds=list(range(P)), device=DEV)
    noise = OUNoise(P * N, device=DEV)
    rep = PopulationReplay(P, 4096, 0, device=DEV)
    rng = np.random.default_rng(0)
    train_population(env, pop, noise, replay=rep, steps=64, collect_steps=64)      # the rings hold min_batch from now on

    def train():
        train_population(env, pop, noise, replay=rep, steps=64, collect_steps=64, reset=False)

    scores = {}

    def evaluate():
        scores["s"] = evaluate_population(env, pop, N, offset=int(rng.integers(0, 2**62))).mean_return.cpu().numpy()

    def exploit():
        dst, src, factors = pbt_plan(scores["s"], 0.25, rng=rng)
        pop.exploit(dst, src)
        table = pop.hyper_table()
        for d, f in zip(dst, factors):
            h = table[d]
            pop.set_hyper(d, actor_lr=h[0] * f[0], critic_lr=h[1] * f[1], tau=h[2] * f[2])
    return {"members": P, "train_envs_per_member": N, "eval_envs_per_member": N, "train_steps": 64, "updates": 64,
            "train_ms": timed(train, 1, reps), "evaluate_ms": timed(evaluate, 1, reps), "exploit_ms": timed(exploit, 1, reps)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_ddpg_eval.json"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("evalbench needs a CUDA device")
    res = {**gpu_info(), "torch": torch.__version__, "evaluation": [], "early_exit": None, "pbt_round": None}
    for P in (1, 16, 148):
        for N in (128, 1024):
            r = bench_eval(P, N, a.reps)
            print(json.dumps(r), flush=True)
            res["evaluation"].append(r)
    res["early_exit"] = bench_early_exit(a.reps)
    print(json.dumps(res["early_exit"]), flush=True)
    res["pbt_round"] = bench_pbt_round(a.reps)
    print(json.dumps(res["pbt_round"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
