"""The reference's 2-D study (main_2d.py with Learning_module_2d) on the device, without the plots.

    python examples/main_flow_2d.py [--steps 1200] [--seed 0]

1. idle run                  -> LearningModule2D.estimateDisturbance
2. learning run, mismatched  -> alpha sweeps [-pi, pi] while f varies; LearningModule2D.learn(px, py, alpha, freq, time)
3. desired / baseline runs   -> a test trajectory with varying (alpha_d, f_d): noise-free with the learned a0, and the
                                mismatched, noisy simulator driven with the same actions
4. corrected actions         -> (alpha, f) for all T control steps from ONE LearningModule2D.predict_batch call
5. corrected run             -> compare the tracking error with and without the GP correction
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mr_rl_b200 import run_sim  # noqa: E402
from mr_rl_b200.learning_module_2d import LearningModule2D  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1200, help="learning-run steps")
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    a0_def, dt, noise_var = 1.5, 0.030, 0.5
    idle = np.zeros((100, 3)); idle[:, 2] = np.arange(100) * dt
    k = np.arange(a.steps)
    learn = np.zeros((a.steps, 3))
    # the velocities are smoothed over 14 frames before the fit (Learning_module_2d.py:48-50), so (alpha, f) must change
    # slowly on that scale: f sweeps [0.1, 5] every ~157 steps while alpha sweeps the circle every 400 steps
    learn[:, 0] = (np.cos(k / 25) + 1) / 2 * 4.9 + 0.1
    learn[:, 1] = (k % 400) / 400 * 2 * np.pi - np.pi
    learn[:, 2] = k * dt
    T = 500
    test = np.zeros((T, 3)); test[:, 2] = np.arange(T) * dt
    test[:, 0] = 2.5 + 1.5 * np.sin(np.arange(T) / 40)                 # f_d in [1, 4]
    test[:, 1] = np.concatenate([np.linspace(0, np.pi / 2, 100), np.linspace(np.pi / 2, -np.pi / 2, 100),
                                 np.linspace(-np.pi / 2, 0, 100), np.linspace(0, np.pi / 8, 100), np.linspace(np.pi / 8, -np.pi, 100)])
    kw = dict(device="cuda:0", noise="philox")
    t0 = time.perf_counter()
    gp = LearningModule2D(device="cuda:0")
    gp.gprX.n_restarts_optimizer = gp.gprY.n_restarts_optimizer = 1
    px, py, _, tm, _ = run_sim(idle, init_pos=np.array([0, 0]), noise_var=noise_var, a0=a0_def, is_mismatched=True, seed=a.seed, **kw)
    gp.estimateDisturbance(px, py, tm)
    px, py, al, tm, fr = run_sim(learn, init_pos=np.array([0, 0]), noise_var=noise_var, a0=a0_def, is_mismatched=True, seed=a.seed + 1, **kw)
    a0_sim = gp.learn(px, py, al, fr, tm)
    t_learn = time.perf_counter() - t0
    print(f"drift D = ({gp.Dx:.3f}, {gp.Dy:.3f}), a0 estimate {a0_sim:.3f}, {len(gp.X)} training points, "
          f"GP kernels {gp.gprX.kernel_} | {gp.gprY.kernel_}  [{t_learn:.1f} s]")

    xd, yd, *_ = run_sim(test, init_pos=np.array([0, 0]), noise_var=0.0, a0=a0_sim, **kw)                 # desired
    xb, yb, *_ = run_sim(test, init_pos=np.array([0, 0]), noise_var=noise_var, a0=a0_def, is_mismatched=True, seed=a.seed + 2, **kw)
    vd = a0_sim * test[:, :1] * np.stack([np.cos(test[:, 1]), np.sin(test[:, 1])], 1)
    vd_dev = torch.as_tensor(vd, device="cuda:0")
    gp.predict_batch(vd_dev[:1])                                                                           # first-launch set-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    X, mux, muy, sgx, sgy, iters, status = gp.predict_batch(vd_dev, return_info=True)                      # all T control steps at once
    torch.cuda.synchronize()
    t_pred = time.perf_counter() - t0
    corrected = test.copy(); corrected[:, 1] = X[:, 0].cpu().numpy(); corrected[:, 0] = X[:, 1].cpu().numpy()
    xl, yl, *_ = run_sim(corrected, init_pos=np.array([0, 0]), noise_var=noise_var, a0=a0_def, is_mismatched=True, seed=a.seed + 2, **kw)
    err_b = np.hypot(xb - xd, yb - yd)
    err_l = np.hypot(xl - xd, yl - yd)
    st = np.bincount(status.cpu().numpy(), minlength=3)
    print(f"corrected (alpha, f) for {T} control steps in {t_pred*1e3:.2f} ms, one predict_batch call "
          f"(passes mean {iters.double().mean():.1f} max {int(iters.max())}; status 0/1/2: {st[0]}/{st[1]}/{st[2]}; "
          f"sigma of the GP: {float(sgx.mean()):.3f}, {float(sgy.mean()):.3f})")
    print(f"final tracking error  baseline {err_b[-1]:.2f}  corrected {err_l[-1]:.2f}   mean  baseline {err_b.mean():.2f}  corrected {err_l.mean():.2f}")


if __name__ == "__main__":
    main()
