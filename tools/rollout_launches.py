"""List the launch configuration of the fused rollout for every action source, one line per case.

    python tools/rollout_launches.py --out OUT_DIR/rollout_launches.txt

One ``VecMREnv.rollout`` launch (K = 2, sigma = 1, Philox noise) per case, recorded with torch.profiler (CUDA
activities): kernel name, grid, block, shared memory (static + dynamic, as the profiler reports it) and registers.
Cases: tensor, broadcast and random actions; the actor on the default 3xFP16, the CUDA-core and the 3xTF32 path; the GP
tracking policy; DDPG collection on the 3xFP16 and the 3xTF32 path; per-env parameter rows with tensor, broadcast and
random actions; the random actions with the mismatched model.  Each at 4096 and 2^20 envs, fp64 and fp32 storage.
Two libraries (MR_LIB_PATH) launch the same kernels the same way when their listings are equal.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mr_rl_b200 import LearningModule, VecMREnv  # noqa: E402
from mr_rl_b200 import _lib as L  # noqa: E402
from mr_rl_b200.ddpg import DDPGLearner, OUNoise, ReplayBuffer, collect  # noqa: E402

DEV = "cuda:0"
K = 2


def tracking_module():
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, WhiteKernel
    g = np.load(os.path.join(ROOT, "tests", "golden", "gp.npz"))
    X = g["X"].reshape(-1, 1)
    gx = GaussianProcessRegressor(kernel=RBF(0.2) + WhiteKernel(0.008), optimizer=None).fit(X, g["yx"])
    gy = GaussianProcessRegressor(kernel=RBF(0.25) + WhiteKernel(0.008), optimizer=None).fit(X, g["yy"])
    lm = LearningModule(device=DEV)
    lm.set_models(gx, gy, *(float(v) for v in g["hyper"]))
    th = np.linspace(0.3, -2.0, K)
    v = lm.a0 * lm.freq * np.stack([np.cos(th), np.sin(th)], 1)
    p = np.vstack([np.zeros(2), np.cumsum(v * 0.030, 0)[:-1]])
    return lm.tracking_policy(np.hstack([p, v]), 2.0)


def cases(n, dtype, policy):
    def env(per_env=False, mism=False):
        e = VecMREnv(n, device=DEV, dtype=dtype, noise="philox", seed=1, auto_reset=True, per_env_params=per_env)
        e.reset(noise_var=1.0, a0=1.0, is_mismatched=mism)
        return e

    acts = torch.rand(K, n, 2, device=DEV, dtype=dtype) * torch.tensor([20.0, 6.28], device=DEV, dtype=dtype)
    row = torch.tensor([[10.0, 1.0]] * K, device=DEV, dtype=dtype)
    actor = DDPGLearner(device=DEV, seed=0).actor

    def collector(e):
        learner, noise, rb = DDPGLearner(device=DEV, seed=0), OUNoise(n, device=DEV), ReplayBuffer(K * n, 0, device=DEV)
        return lambda: collect(e, learner, noise, rb, K)

    def with_path(path, fn):
        def run():
            old = L.set_actor_path(path)
            try:
                fn()
            finally:
                L.set_actor_path(old)
        return run

    e = env()
    yield "tensor", e, lambda: e.rollout(actions=acts)
    yield "broadcast", e, lambda: e.rollout(actions=row)
    yield "random", e, lambda: e.rollout(policy="random", k_steps=K)
    yield "actor_fp16", e, lambda: e.rollout(policy=actor, k_steps=K)
    yield "actor_simt", e, with_path("simt", lambda: e.rollout(policy=actor, k_steps=K))
    yield "actor_tf32", e, with_path("tf32", lambda: e.rollout(policy=actor, k_steps=K))
    yield "gp_tracking", e, lambda: e.rollout(policy=policy)
    yield "collect_fp16", e, collector(e)
    yield "collect_tf32", e, with_path("tf32", collector(e))
    em = env(mism=True)
    yield "random_mismatched", em, lambda: em.rollout(policy="random", k_steps=K)
    ep = env(per_env=True)
    yield "per_env_tensor", ep, lambda: ep.rollout(actions=acts)
    yield "per_env_broadcast", ep, lambda: ep.rollout(actions=row)
    yield "per_env_random", ep, lambda: ep.rollout(policy="random", k_steps=K)


def launches(fn):
    fn()                                                     # warm-up: module load and kernel attributes
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    path = os.path.join(OUT_DIR, "_trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    os.remove(path)
    return [f"{ev['name']} grid={ev['args']['grid']} block={ev['args']['block']} "
            f"smem={ev['args']['shared memory']} regs={ev['args']['registers per thread']}"
            for ev in sorted(events, key=lambda ev: ev.get("ts", 0))
            if ev.get("cat") == "kernel" and "env_rollout_kernel" in ev["name"]]


def main():
    global OUT_DIR
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="the listing; the profiler trace is written beside it and removed")
    a = ap.parse_args()
    OUT_DIR = os.path.dirname(os.path.abspath(a.out))
    os.makedirs(OUT_DIR, exist_ok=True)
    policy = tracking_module()
    lines = []
    for dtype in (torch.float64, torch.float32):
        for n in (4096, 1 << 20):
            for name, env, fn in cases(n, dtype, policy):
                for k in launches(fn):
                    lines.append(f"{str(dtype)[6:]} n={n} {name}: {k}")
                env.check_status()
            torch.cuda.empty_cache()
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print(f"{len(lines)} launches -> {a.out}")


if __name__ == "__main__":
    main()
