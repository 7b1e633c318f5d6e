"""A DDPG hyper-parameter sweep as ONE population: actor / critic learning rates x seeds, every member a complete learner
with its own envs, OU noise and replay ring, all trained together (one collect launch and one update launch per step for
the whole population).

    python examples/ddpg_sweep.py [--envs-per-member 1024] [--steps 640] [--collect-steps 64] [--seeds 4]

Member p equals the solo run train(collect_steps=K) of DDPGLearner(seed, actor_lr, critic_lr) on envs p N .. p N + N - 1.
The shaped reward (calculate_reward, MR_env.py:118-134) gives the members something to tell apart.  After training, every
member's greedy policy plays --eval-envs fresh episodes (one evaluate_population launch, common random numbers), and that
return is printed beside the training reward (which mixes in the exploration noise and spans a changing policy).
"""
import argparse
import itertools
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from mr_rl_b200 import DDPGPopulation, OUNoise, PopulationReplay, VecMREnv
from mr_rl_b200.ddpg import evaluate_population, train_population


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs-per-member", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=640)
    ap.add_argument("--collect-steps", type=int, default=64)
    ap.add_argument("--seeds", type=int, default=4)
    ap.add_argument("--eval-envs", type=int, default=1024)
    ap.add_argument("--actor-lr", type=float, nargs="*", default=[1e-4, 3e-4, 1e-3, 3e-3])
    ap.add_argument("--critic-lr", type=float, nargs="*", default=[1e-3, 3e-3, 1e-2, 3e-2])
    args = ap.parse_args()
    dev = "cuda:0"
    grid = list(itertools.product(args.actor_lr, args.critic_lr, range(args.seeds)))
    P, N = len(grid), args.envs_per_member
    env = VecMREnv(P * N, device=dev, noise="philox", seed=0, auto_reset=True, reward_mode="shaped")
    pop = DDPGPopulation(P, seeds=[s for _, _, s in grid], actor_lr=[a for a, _, _ in grid], critic_lr=[c for _, c, _ in grid],
                         device=dev)
    replay = PopulationReplay(P, max(10000, 8 * N), device=dev)
    t0 = time.perf_counter()
    log = train_population(env, pop, OUNoise(P * N, device=dev), min_batch=64, steps=args.steps, replay=replay,
                           collect_steps=args.collect_steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    launches = log.shape[1]
    stats = pop.stats.cpu().numpy()
    print(f"{P} members x {N} envs, {args.steps} env steps, {pop.updates} updates per member: {dt:.2f} s, "
          f"{dt / launches * 1e3:.1f} ms per iteration (collect {args.collect_steps} steps + {args.collect_steps} updates)")
    t0 = time.perf_counter()
    ev = evaluate_population(env, pop, args.eval_envs)
    greedy, goal = ev.mean_return.cpu().numpy(), ev.goal_rate.cpu().numpy()
    print(f"greedy evaluation, {args.eval_envs} episodes per member: {(time.perf_counter() - t0) * 1e3:.1f} ms")
    print(" actor_lr critic_lr seed   final mean reward   mean episode reward   greedy return   goal rate")
    for p, (a, c, s) in enumerate(grid):
        ep = stats[p, 0]
        per_ep = stats[p, 2] / ep if ep else float("nan")
        print(f"{a:9.0e} {c:9.0e} {s:4d}   {log[p, -1, 0]:17.4f}   {per_ep:19.3f}   {greedy[p]:13.3f}   {goal[p]:9.3f}")
    env.check_status()


if __name__ == "__main__":
    main()
