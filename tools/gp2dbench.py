"""Time LearningModule2D.predict_batch's search (mr_gp_correct_action_2d) on the GPU.

    python tools/gp2dbench.py [--out profiles/r03_gp2d_predict.json] [--reps 20]

Models: the golden 2-D model (tests/golden/learn_2d.npz at its fitted theta, n_train = 272) and a synthetic one with
n_train = 2048 (inputs over [-pi, pi] x [0.1, 5], smooth targets, fixed hyper-parameters).  Velocities: N = 4096 and
N = 262 144 desired velocities of the interior regime (alpha_d in [-pi + 0.5, pi - 0.5], f_d in [1, 3.5]).  Per case:
CUDA events around ``--reps`` launches after a warm-up; ms per call, velocities/s, passes, and kernel evaluations/s =
2 n_train sum(passes) / time (each pass evaluates both GPs at every training point).  The model (<= 100 KB) stays in
L1/L2, so the search is FP64-pipe bound like the 1-D mean kernel.  Host baseline: LearningModule2D.predict (scipy
minimize, two mr_gp_predict launches and a device sync per objective evaluation) over 32 velocities, wall clock.
The GPU's name and power limit are read in the same run (read-only nvidia-smi query).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mr_rl_b200 import _lib as L  # noqa: E402
from mr_rl_b200.learning_module_2d import LearningModule2D  # noqa: E402

MEAN_1D_EVALS_PER_S = 7.9e11      # DESIGN §4.3: the staged 1-D mean kernel, 262 144 queries x 2000 points, one GP


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def models():
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, WhiteKernel
    z = np.load(os.path.join(ROOT, "tests", "golden", "learn_2d.npz"))
    fit = lambda X, y, ls, noise: GaussianProcessRegressor(RBF(ls) + WhiteKernel(noise), optimizer=None).fit(X, y)
    th_x, th_y = z["theta_x"], z["theta_y"]
    yield "golden_n272", fit(z["X"], z["Yx"], *np.exp(th_x)), fit(z["X"], z["Yy"], *np.exp(th_y)), float(z["a0"])
    rng = np.random.default_rng(5)
    n = 2048
    X = np.stack([rng.uniform(-np.pi, np.pi, n), rng.uniform(0.1, 5.0, n)], 1)
    yx = 0.4 * np.sin(X[:, 0]) * np.exp(-0.2 * X[:, 1]) + 0.1 * np.cos(0.7 * X[:, 1]) + 0.02 * rng.standard_normal(n)
    yy = -0.3 * np.cos(X[:, 0] + 0.5) + 0.05 * X[:, 1] + 0.02 * rng.standard_normal(n)
    yield "synthetic_n2048", fit(X, yx, 0.8, 4e-4), fit(X, yy, 0.9, 4e-4), 2.0


def interior(n, a0, seed):
    rng = np.random.default_rng(seed)
    ad, fd = rng.uniform(-np.pi + 0.5, np.pi - 0.5, n), rng.uniform(1.0, 3.5, n)
    return a0 * fd[:, None] * np.stack([np.cos(ad), np.sin(ad)], 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_gp2d_predict.json"))
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    lib = L.load()
    dev = torch.device("cuda:0")
    result = {"what": "mr_gp_correct_action_2d (LearningModule2D.predict_batch's search), interior regime", **gpu_info(),
              "mean_1d_kernel_evals_per_s": MEAN_1D_EVALS_PER_S, "cases": []}
    lo, hi = (C.c_double * 2)(-np.pi, 0.0), (C.c_double * 2)(np.pi, 5.0)
    for name, gx, gy, a0 in models():
        lm = LearningModule2D(device="cuda:0", fit="host")
        lm.set_models(gx, gy, a0)
        n_train = lm._dx.n_train
        for N in (4096, 262144):
            vd = torch.as_tensor(interior(N, a0, seed=N), device=dev).contiguous()
            X = torch.empty((N, 2), dtype=torch.float64, device=dev)
            it = torch.empty(N, dtype=torch.int32, device=dev)
            st = torch.empty(N, dtype=torch.uint8, device=dev)
            call = lambda: lib.mr_gp_correct_action_2d(C.byref(lm._dx._c), C.byref(lm._dy._c), vd.data_ptr(), N, float(a0), lo, hi,
                                                       X.data_ptr(), it.data_ptr(), st.data_ptr(), None)
            for _ in range(3):
                L.check(call(), "mr_gp_correct_action_2d")
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                call()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.reps
            passes = it.double()
            evals = 2.0 * n_train * float(passes.sum())
            t0 = time.perf_counter()
            lm.predict_batch(vd)
            torch.cuda.synchronize()
            row = {"model": name, "n_train": n_train, "n_velocities": N, "ms_per_call": ms, "velocities_per_s": N / ms * 1e3,
                   "passes_mean": float(passes.mean()), "passes_max": int(it.max()),
                   "status_counts": np.bincount(st.cpu().numpy(), minlength=3).tolist(),
                   "kernel_evals_per_s": evals / ms * 1e3, "ratio_to_1d_mean_kernel": evals / ms * 1e3 / MEAN_1D_EVALS_PER_S,
                   "predict_batch_with_posterior_ms_wall": (time.perf_counter() - t0) * 1e3}
            result["cases"].append(row)
            print(json.dumps(row), flush=True)
        # host path: scipy minimize with the device GPs in the loop, one velocity at a time
        vd = interior(32, a0, seed=99)
        lm.predict(vd[0])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for v in vd:
            lm.predict(v)
        torch.cuda.synchronize()
        host_ms = (time.perf_counter() - t0) * 1e3 / len(vd)
        best = max((c for c in result["cases"] if c["model"] == name), key=lambda c: c["velocities_per_s"])
        row = {"model": name, "host_predict_ms_per_velocity": host_ms, "host_velocities": len(vd),
               "speedup_per_velocity": host_ms * 1e-3 * best["velocities_per_s"]}
        result["cases"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "cases"}))


if __name__ == "__main__":
    main()
