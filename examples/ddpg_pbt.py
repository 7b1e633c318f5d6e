"""Population-based training of DDPG learners: train the population, evaluate every member's greedy policy in one launch,
copy the best members over the worst and perturb the copies' learning rates and tau, repeat.

    python examples/ddpg_pbt.py [--members 64] [--envs-per-member 1024] [--rounds 5] [--steps-per-round 128]
                                [--eval-envs 1024] [--fraction 0.25] [--seed 0]

The members start from a grid of actor / critic learning rates.  The ranking is the mean return of --eval-envs greedy
episodes per member with common random numbers (every member meets the same starts and noise), on the shaped reward
(calculate_reward, MR_env.py:118-134).
"""
import argparse
import itertools
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from mr_rl_b200 import DDPGPopulation, OUNoise, PopulationReplay, VecMREnv
from mr_rl_b200.ddpg import pbt_population


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--members", type=int, default=64)
    ap.add_argument("--envs-per-member", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps-per-round", type=int, default=128)
    ap.add_argument("--collect-steps", type=int, default=64)
    ap.add_argument("--eval-envs", type=int, default=1024)
    ap.add_argument("--fraction", type=float, default=0.25)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    dev = "cuda:0"
    P, N = args.members, args.envs_per_member
    grid = list(itertools.islice(itertools.cycle(itertools.product([1e-4, 3e-4, 1e-3, 3e-3], [1e-3, 3e-3, 1e-2, 3e-2])), P))
    env = VecMREnv(P * N, device=dev, noise="philox", seed=args.seed, auto_reset=True, reward_mode="shaped")
    pop = DDPGPopulation(P, seeds=list(range(P)), actor_lr=[a for a, _ in grid], critic_lr=[c for _, c in grid], device=dev)
    replay = PopulationReplay(P, max(10000, 8 * N), device=dev)
    t0 = time.perf_counter()
    hist = pbt_population(env, pop, OUNoise(P * N, device=dev), replay, args.rounds, args.steps_per_round, args.eval_envs,
                          fraction=args.fraction, seed=args.seed, collect_steps=args.collect_steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    print(f"{P} members x {N} envs, {args.rounds} rounds of {args.steps_per_round} env steps: {dt:.2f} s")
    print("round   best return   median return   replaced   best member (actor_lr, critic_lr, tau)")
    for r in range(args.rounds):
        s = hist["score"][r]
        b = int(np.argmax(s))
        h = hist["hyper"][r, b]
        replaced = int((hist["parent"][r] != np.arange(P)).sum())
        print(f"{r:5d}   {s[b]:11.3f}   {np.median(s):13.3f}   {replaced:8d}   {b:4d} ({h[0]:.2e}, {h[1]:.2e}, {h[2]:.2e})")
    env.check_status()


if __name__ == "__main__":
    main()
