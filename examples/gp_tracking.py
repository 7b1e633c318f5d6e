"""GP-corrected tracking over many noise realisations, one launch per controller.

    python examples/gp_tracking.py [--envs 4096] [--gain 2.0] [--steps 600] [--goal]

1. idle run, learning run, desired run (main_flow.py steps 1-3; main.py:56-75,119-131)
2. on N envs (independent Philox noise per env, mismatched simulator), one fused rollout each for
   - the uncorrected baseline: main.py's desired actions broadcast to every env;
   - the open-loop correction (gain 0): main.py's corrected run, vd = desired velocity;
   - the closed-loop correction: vd = desired velocity + gain * (desired position - position), per env and step.
   Prints the mean / median / 95th-percentile tracking error against the desired path and the time of each launch.
--goal: go-to-goal with the closed-loop controller (reference = the origin, auto reset on), episode statistics.
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mr_rl_b200 import LearningModule, VecMREnv, run_sim  # noqa: E402


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--gain", type=float, default=2.0, help="position feedback of the closed-loop run, 1/s")
    ap.add_argument("--steps", type=int, default=600, help="training steps of the learning run")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--goal", action="store_true", help="go-to-goal with auto reset instead of path tracking")
    a = ap.parse_args()
    freq, a0_def, dt, noise_var = 4.0, 1.5, 0.030, 0.5                 # main.py:9-11,53
    idle = np.zeros((100, 3)); idle[:, 2] = np.arange(100) * dt
    cyc = a.steps // 3
    circle = np.zeros((cyc, 3)); circle[:, 0] = freq; circle[:, 1] = np.linspace(-np.pi, np.pi, cyc)
    learn = np.vstack([circle] * 3); learn[:, 2] = np.arange(len(learn)) * dt
    T = 500
    test = np.zeros((T, 3)); test[:, 0] = freq; test[:, 2] = np.arange(T) * dt
    test[:, 1] = np.concatenate([np.linspace(0, np.pi / 2, 100), np.linspace(np.pi / 2, -np.pi / 2, 100),
                                 np.linspace(-np.pi / 2, 0, 100), np.linspace(0, np.pi / 8, 100), np.linspace(np.pi / 8, -np.pi, 100)])
    kw = dict(device="cuda:0", noise="philox")
    gp = LearningModule(device="cuda:0")
    gp.gprX.n_restarts_optimizer = gp.gprY.n_restarts_optimizer = 1
    px, py, _, tm, _ = run_sim(idle, init_pos=np.array([0, 0]), noise_var=noise_var, a0=a0_def, is_mismatched=True, seed=a.seed, **kw)
    gp.estimateDisturbance(px, py, tm)
    px, py, al, tm, _ = run_sim(learn, init_pos=np.array([0, 0]), noise_var=noise_var, a0=a0_def, is_mismatched=True, seed=a.seed + 1, **kw)
    a0_sim = gp.learn(px, py, al, tm, learn)
    print(f"drift D = ({gp.Dx:.3f}, {gp.Dy:.3f}), a0 estimate {a0_sim:.3f}, heading surrogate "
          f"{'accepted' if gp._cheb is not None else 'refused'}")
    xd, yd, *_ = run_sim(test, init_pos=np.array([0, 0]), noise_var=0.0, a0=a0_sim, **kw)                 # desired
    # ref[k] = (desired position at the start of step k, desired velocity during it), main.py:147
    start = np.vstack([[0.0, 0.0], np.stack([xd, yd], 1)[:-1]])
    ref = np.hstack([start, a0_sim * freq * np.stack([np.cos(test[:, 1]), np.sin(test[:, 1])], 1)])
    n = a.envs

    def env_at_origin(**ekw):
        e = VecMREnv(n, device="cuda:0", noise="philox", seed=a.seed + 2, **ekw)
        e.reset(init=np.zeros(2), noise_var=noise_var, a0=a0_def, is_mismatched=True)
        return e

    if a.goal:
        e = env_at_origin(auto_reset=True)
        e.init_space.low[:] = -150.0; e.init_space.high[:] = 150.0; e.init_space = e.init_space
        e.reset(init=None, noise_var=noise_var, a0=a0_def, is_mismatched=True)
        goal = np.zeros((T, 4))                                         # reference = the origin, no feed-forward velocity
        _, ms = timed(lambda: e.rollout(policy=gp.tracking_policy(goal, a.gain)))
        s = e.stats_dict()
        print(f"go-to-goal, {n} envs x {T} steps, gain {a.gain}: {s['episodes']:.0f} episodes, goal rate "
              f"{s['goal'] / max(s['episodes'], 1):.3f}, out of bounds {s['out_of_bounds']:.0f}, timeouts {s['timeout']:.0f}, "
              f"mean length {s['mean_episode_length']:.1f} steps  [{ms:.1f} ms]")
        return

    desired = torch.as_tensor(np.stack([xd, yd], 0), device="cuda:0")[:, :, None]          # [2, T, 1]
    runs = {"baseline": lambda e: e.rollout(actions=torch.as_tensor(test[:, :2]), record=True),
            "open loop (gain 0)": lambda e: e.rollout(policy=gp.tracking_policy(ref, 0.0), record=True),
            f"closed loop (gain {a.gain:g})": lambda e: e.rollout(policy=gp.tracking_policy(ref, a.gain), record=True)}
    print(f"tracking error against the desired path, {n} envs x {T} steps (sigma {noise_var}, mismatched):")
    for name, run in runs.items():
        e = env_at_origin()
        run(e)                                                          # warm-up (module load)
        e = env_at_origin()
        res, ms = timed(lambda: run(e))
        xy = res["xy"].permute(1, 0, 2)                                 # [2, T, N]
        err = torch.sqrt(((xy - desired) ** 2).sum(0))                  # [T, N]
        per_env = err.mean(0)
        q = torch.quantile(per_env, torch.tensor([0.5, 0.95], device=per_env.device, dtype=per_env.dtype)).tolist()
        fin = err[-1]
        print(f"  {name:22s} mean {float(per_env.mean()):7.2f}  median {q[0]:7.2f}  p95 {q[1]:7.2f}   "
              f"final: mean {float(fin.mean()):7.2f}  p95 {float(torch.quantile(fin, 0.95)):7.2f}   [{ms:.2f} ms]")
        e.check_status()


if __name__ == "__main__":
    main()
