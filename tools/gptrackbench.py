"""Time the GP-corrected heading controller: the fused policy rollout against the composed control loop.

    python tools/gptrackbench.py [--out profiles/r04_gp_tracking.json] [--gain 2.0]

Fused: one ``VecMREnv.rollout(policy=LearningModule.tracking_policy(ref, gain))`` launch (mr_env_rollout_gp_heading) for
K steps.  Composed: per step, vd = ref[k, 2:] + gain * (ref[k, :2] - last_pos) in torch (3 launches), the standalone
heading search mr_gp_correct_heading_cheb called directly (no posterior), the heading copied into the action rows and one
``env.step``: 6 launches and a round trip of state, vd and actions through HBM per step.  Both start from the same state
and must end in the same state bit for bit (reported).

Sizes: 4096 envs x K = 500 (main.py's trajectory length, batched) and 2^20 envs x K = 64.  Simulator: sigma = 0.5,
mismatched model, Philox noise, a0 = 1.5.  Models: the golden GP (tests/golden/gp.npz, RBF 0.2 / 0.25) and a synthetic one
with 2000 training points.  Timing: CUDA events around each launch sequence after a warm-up of both paths, the state
restored between repetitions outside the timed window; the best of ``--reps``.  Objective evaluations per step come from
an untimed composed run with the standalone kernel's nfev output.  The GPU's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mr_rl_b200 import LearningModule, VecMREnv  # noqa: E402
from mr_rl_b200 import _lib as L  # noqa: E402

DEV = "cuda:0"
A0_SIM, SIGMA = 1.5, 0.5


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"gpu": name.strip(), "power_limit": power.strip()}


def models():
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, WhiteKernel
    g = np.load(os.path.join(ROOT, "tests", "golden", "gp.npz"))
    X = g["X"].reshape(-1, 1)
    fit = lambda X, y, ls, noise: GaussianProcessRegressor(kernel=RBF(ls) + WhiteKernel(noise), optimizer=None).fit(X, y)
    yield f"golden_n{len(X)}", fit(X, g["yx"], 0.2, 0.008), fit(X, g["yy"], 0.25, 0.008), tuple(float(v) for v in g["hyper"])
    rng = np.random.default_rng(11)
    n = 2000
    X = rng.uniform(-np.pi, np.pi, (n, 1))
    yx = 0.3 * np.sin(X[:, 0]) + 0.1 * np.cos(3 * X[:, 0]) + 0.02 * rng.standard_normal(n)
    yy = -0.25 * np.cos(X[:, 0] + 0.4) + 0.05 * np.sin(2 * X[:, 0]) + 0.02 * rng.standard_normal(n)
    yield "synthetic_n2000", fit(X, yx, 0.3, 4e-4), fit(X, yy, 0.3, 4e-4), (1.4, 4.0, 0.21, -0.12)


def desired_ref(lm, K):
    """main_flow's desired heading schedule (five sweeps), fixed speed a0 freq, positions accumulated over dt."""
    th = np.concatenate([np.linspace(0, np.pi / 2, 100), np.linspace(np.pi / 2, -np.pi / 2, 100), np.linspace(-np.pi / 2, 0, 100),
                         np.linspace(0, np.pi / 8, 100), np.linspace(np.pi / 8, -np.pi, 100)])[:K]
    v = lm.a0 * lm.freq * np.stack([np.cos(th), np.sin(th)], 1)
    p = np.vstack([np.zeros(2), np.cumsum(v * 0.030, 0)[:-1]])
    return np.hstack([p, v])


class Composed:
    """The hand-built control loop with the standalone search called directly (no posterior)."""

    def __init__(self, lm, env, ref, gain):
        self.lm, self.env, self.gain = lm, env, gain
        self.ref = torch.as_tensor(ref, device=DEV)
        n = env.num_envs
        self.alpha = torch.empty(n, dtype=torch.float64, device=DEV)
        self.act = torch.full((n, 2), float(lm.freq), dtype=torch.float64, device=DEV)
        self.lib = L.load()

    def run(self, K, nfev=None):
        lm, env, cheb = self.lm, self.env, self.lm._cheb
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        total = 0
        for k in range(K):
            vd = (self.ref[k, 2:] + self.gain * (self.ref[k, :2] - env.last_pos)).contiguous()
            rc = self.lib.mr_gp_correct_heading_cheb(cheb[0].data_ptr(), cheb[1].data_ptr(), cheb.shape[1], vd.data_ptr(),
                                                     env.num_envs, float(lm.a0), float(lm.freq), float(lm.Dx), float(lm.Dy),
                                                     self.alpha.data_ptr(), nfev.data_ptr() if nfev is not None else None, stream)
            L.check(rc, "mr_gp_correct_heading_cheb")
            if nfev is not None:
                total += int(nfev.sum())
            self.act[:, 1].copy_(self.alpha)
            env.step(self.act)
        return total


def snapshot(env):
    return [t.clone() for t in (env._state, env._counter, env._status, env._cursor)], env._step_index


def restore(env, snap):
    for t, s in zip((env._state, env._counter, env._status, env._cursor), snap[0]):
        t.copy_(s)
    env._step_index = snap[1]


def timed(fn, reps, env, snap):
    best = float("inf")
    for _ in range(reps):
        restore(env, snap)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def case(lm, name, n, K, gain, reps):
    ref = desired_ref(lm, K)
    env = VecMREnv(n, device=DEV, noise="philox", seed=3)
    rng = np.random.default_rng(n)
    env.reset(init=rng.uniform(-2, 2, (n, 2)), noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
    snap = snapshot(env)
    pol = lm.tracking_policy(ref, gain)
    comp = Composed(lm, env, ref, gain)
    fused = lambda: env.rollout(policy=pol, accumulate_stats=False)
    restore(env, snap); fused(); restore(env, snap); comp.run(min(K, 8))      # warm-up of both paths
    ms_fused = timed(fused, reps, env, snap)
    end_fused = [t.clone() for t in (env._state, env._counter, env._status)]
    ms_comp = timed(lambda: comp.run(K), max(1, reps // 2), env, snap)
    end_comp = [t.clone() for t in (env._state, env._counter, env._status)]
    same = all(torch.equal(a, b) for a, b in zip(end_fused, end_comp))
    restore(env, snap)
    nfev = torch.empty(n, dtype=torch.int32, device=DEV)
    evals = comp.run(K, nfev)
    row = {"model": name, "n_coef": int(lm._cheb.shape[1]), "envs": n, "k_steps": K, "gain": gain,
           "fused_ms": ms_fused, "fused_env_steps_per_s": n * K / ms_fused * 1e3,
           "composed_ms": ms_comp, "composed_env_steps_per_s": n * K / ms_comp * 1e3, "fused_speedup": ms_comp / ms_fused,
           "objective_evals_per_env_step": evals / (n * K), "final_state_bit_identical": same,
           "status_flags_set": int((env.status != 0).sum())}
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_gp_tracking.json"))
    ap.add_argument("--gain", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=4)
    a = ap.parse_args()
    result = {"what": "GP-corrected heading control: fused policy rollout (mr_env_rollout_gp_heading) vs composed loop "
                      "(torch vd, mr_gp_correct_heading_cheb, env.step); sigma 0.5, mismatched, Philox noise",
              **gpu_info(), "cases": []}
    for name, gx, gy, (a0, freq, dx, dy) in models():
        lm = LearningModule(device=DEV)
        lm.set_models(gx, gy, a0, freq, dx, dy)
        if lm._cheb is None:
            result["cases"].append({"model": name, "skipped": "heading surrogate not accepted"})
            continue
        for n, K in ((4096, 500), (1 << 20, 64)):
            result["cases"].append(case(lm, name, n, K, a.gain, a.reps))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "cases"}))


if __name__ == "__main__":
    main()
