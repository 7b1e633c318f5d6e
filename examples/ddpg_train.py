"""The learner of RL/MR_ddpg.py on the device: N envs act with mu(s) + OU noise, every transition enters a replay ring in
HBM, one kernel launch per learner update (critic + actor + targets).

    python examples/ddpg_train.py [--envs 4096] [--iters 500] [--batch 64] [--reward shaped] [--collect-steps 64]

With the reference's constant reward (10 per step, MR_env.py:89) there is nothing to learn but the value scale; the
shaped reward (calculate_reward, MR_env.py:118-134, defined but unused upstream) is offered for experiments.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from mr_rl_b200 import DDPGLearner, OUNoise, ReplayBuffer, VecMREnv
from mr_rl_b200.ddpg import train


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--iters", type=int, default=500)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--updates-per-step", type=int, default=1)
    ap.add_argument("--reward", choices=["const", "shaped"], default="const")
    ap.add_argument("--collect-steps", type=int, default=None,
                    help="K env steps per fused collection launch (ddpg.collect), then K * updates-per-step updates")
    args = ap.parse_args()
    dev = "cuda:0"
    env = VecMREnv(args.envs, device=dev, noise="philox", seed=0, auto_reset=True, reward_mode=args.reward)
    learner = DDPGLearner(device=dev, seed=0)                     # actor 1e-3, critic 1e-2, tau 1e-3, gamma 0.99 (:337-341)
    replay = ReplayBuffer(max(10000, 8 * args.envs), 0, device=dev)
    noise = OUNoise(args.envs, device=dev)
    t0 = time.perf_counter()
    log = train(env, learner, noise, min_batch=args.batch, steps=args.iters, updates_per_step=args.updates_per_step,
                replay=replay, log_every=max(1, args.iters // (10 * (args.collect_steps or 1))),
                collect_steps=args.collect_steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    print(f"{args.iters} iterations x {args.envs} envs in {dt:.2f} s: {args.iters * args.envs / dt:.3g} env-steps/s, "
          f"{learner.updates} learner updates ({learner.updates / dt:.0f}/s), final critic loss {log[-1, 1]:.4g}")
    env.check_status()


if __name__ == "__main__":
    main()
