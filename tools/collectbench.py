"""Time DDPG experience collection: the fused collector (ddpg.collect) against the composed acting loop of ddpg.train.

    python tools/collectbench.py [--out profiles/r05_ddpg_collect.json] [--reps 3]

Collection, K = 64 env steps at 4096, 65 536 and 2^20 envs (sigma = 1, Philox noise, auto reset, default 3xFP16 actor path
unless noted):
  composed  per step learner.predict -> OUNoise.add_to -> env.step -> ReplayBuffer.add (four launches) and the state copy
  fused     one ddpg.collect launch (mr_env_rollout_ddpg_collect), also with the 3xTF32 actor path
  rollout   the plain actor rollout (VecMREnv.rollout(policy=actor)): no OU noise, no ring writes
The ring holds K n transitions, so the fused launch writes every one of them (56 bytes each).

Training: ddpg.train() against train(collect_steps=64), same ratio of one update per env step, at 4096 envs with batch 64
and at 2^20 envs with batch 65 536, 128 env steps each.  The same loops are also run with CUDA events between the
collection and the learner phases, which splits each iteration's time in two.

Timing: CUDA events after a warm-up of every path, the best of --reps.  The GPU's name and power limit are read in the
same run.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mr_rl_b200 import VecMREnv  # noqa: E402
from mr_rl_b200 import _lib as L  # noqa: E402
from mr_rl_b200.ddpg import DDPGLearner, OUNoise, ReplayBuffer, collect, train  # noqa: E402

DEV = "cuda:0"
K = 64
RING_BYTES = (5 + 2 + 1 + 1 + 5) * 4


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def make(n, capacity):
    env = VecMREnv(n, device=DEV, noise="philox", seed=1, auto_reset=True)
    env.reset(noise_var=1.0, a0=1.0)
    return env, DDPGLearner(device=DEV, seed=0), OUNoise(n, device=DEV), ReplayBuffer(capacity, 0, device=DEV)


def composed_steps(env, learner, noise, rb, k, state):
    n = env.num_envs
    for _ in range(k):
        a = learner.predict(state, n)
        noise.add_to(a)
        _, rew, done, _ = env.step(a)
        rb.add(state, a, rew, done, env._obs, n)
        state.copy_(env._obs)


def best_ms(fn, reps):
    best = math.inf
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def collection_case(n, reps):
    env, learner, noise, rb = make(n, K * n)
    state = env._obs.clone()
    comp = lambda: composed_steps(env, learner, noise, rb, K, state)
    fused = lambda: collect(env, learner, noise, rb, K)
    plain = lambda: env.rollout(policy=learner.actor, k_steps=K)
    for f in (comp, fused, plain):
        f()
    row = {"envs": n, "k_steps": K}
    ms = {"composed": best_ms(comp, reps), "fused_fp16": best_ms(fused, reps), "actor_rollout_fp16": best_ms(plain, reps)}
    old = L.set_actor_path("tf32")
    try:
        fused(); plain()
        ms["fused_tf32"] = best_ms(fused, reps)
        ms["actor_rollout_tf32"] = best_ms(plain, reps)
    finally:
        L.set_actor_path(old)
    env.check_status()
    for k, v in ms.items():
        row[f"{k}_ms"] = v
        row[f"{k}_env_steps_per_s"] = n * K / v * 1e3
    row["fused_speedup_over_composed"] = ms["composed"] / ms["fused_fp16"]
    row["fused_cost_over_actor_rollout"] = ms["fused_fp16"] / ms["actor_rollout_fp16"]
    row["fused_ring_bytes_per_s"] = n * K * RING_BYTES / ms["fused_fp16"] * 1e3
    print(json.dumps(row), flush=True)
    del env, learner, noise, rb, state
    torch.cuda.empty_cache()
    return row


def split_loop(n, batch, steps, collect_steps):
    """train()'s loop with CUDA events between collection and learner; returns (collection ms, learner ms, total ms)."""
    env, learner, noise, rb = make(n, K * n)
    state = env._obs.clone()
    marks = []
    k = collect_steps or 1
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for it in range(steps // k):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        if collect_steps:
            collect(env, learner, noise, rb, k)
        else:
            composed_steps(env, learner, noise, rb, 1, state)
        ev[1].record()
        if rb.size() >= batch:
            for _ in range(k):
                learner.update(rb, batch)
        ev[2].record()
        marks.append(ev)
    torch.cuda.synchronize()
    total = (time.perf_counter() - t0) * 1e3
    col = sum(e[0].elapsed_time(e[1]) for e in marks)
    lrn = sum(e[1].elapsed_time(e[2]) for e in marks)
    return col, lrn, total


def training_case(n, batch, steps, reps):
    row = {"envs": n, "batch": batch, "env_steps_per_env": steps, "updates": steps}
    for label, cs in (("train", None), ("train_collect64", K)):
        env, learner, noise, rb = make(n, K * n)
        run = lambda: train(env, learner, noise, min_batch=batch, steps=steps, replay=rb, collect_steps=cs)
        run()                                                          # warm-up
        best = math.inf
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run()
            torch.cuda.synchronize()
            best = min(best, (time.perf_counter() - t0) * 1e3)
        row[f"{label}_ms"] = best
        row[f"{label}_env_steps_per_s"] = n * steps / best * 1e3
        del env, learner, noise, rb
        torch.cuda.empty_cache()
        split_loop(n, batch, K, cs)                                    # warm-up
        col, lrn, tot = min((split_loop(n, batch, steps, cs) for _ in range(reps)), key=lambda r: r[2])
        row[f"{label}_split_collection_ms"] = col
        row[f"{label}_split_learner_ms"] = lrn
        row[f"{label}_split_collection_share"] = col / (col + lrn)
        torch.cuda.empty_cache()
    row["train_speedup"] = row["train_ms"] / row["train_collect64_ms"]
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_ddpg_collect.json"))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    result = {"what": "DDPG experience collection: fused collector (mr_env_rollout_ddpg_collect) vs the composed loop "
                      "(actor, OU noise, env step, replay add per step) vs the plain actor rollout; sigma 1, Philox noise, "
                      f"auto reset, K = {K}; and ddpg.train() vs train(collect_steps={K})",
              **gpu_info(), "collection": [], "training": []}
    for n in (4096, 65536, 1 << 20):
        result["collection"].append(collection_case(n, a.reps))
    for n, batch in ((4096, 64), (1 << 20, 65536)):
        result["training"].append(training_case(n, batch, 2 * K, a.reps))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k not in ("collection", "training")}))


if __name__ == "__main__":
    main()
