"""Dev tool: time the single-step / rollout kernels for a few configurations (CUDA events).

    python tools/stepbench.py [--n 1048576] [--steps 200] [--rollout]
    python tools/stepbench.py --ab LIB_A LIB_B [LIB_C ...] [--rounds 5] [--bench] [--rollout]

--ab runs the same measurements for two or more builds of the library (python -m mr_rl_b200.build --variant=X writes
mr_rl_b200/_lib/libmr_rl_b200X.so), each in a fresh subprocess with MR_LIB_PATH pointing at it, alternating A, B, A, B ...
(the order reverses every round) for --rounds rounds, and prints the median and min-max of every configuration per
library, and each library's median over A's.  --bench adds the bench.py headline (`value`, env-steps/s) to every
round.  Alternating in one session keeps clock and neighbour effects on the shared GPU out of the comparison as far as
possible; the min-max spread says how far they reach.
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BYTES = {"float64": 153, "float32": 81}


def time_step(n, dtype, sigma, steps, auto_reset=True, sp=False):
    import numpy as np
    import torch
    from mr_rl_b200 import VecMREnv
    env = VecMREnv(n, device="cuda:0", dtype=dtype, noise="philox" if sigma else "none", seed=1, auto_reset=auto_reset)
    env.want_state_prime = sp
    env.reset(init=None, noise_var=sigma, a0=1.0)
    acts = torch.rand(8, n, 2, device="cuda:0", dtype=torch.float64)
    acts[..., 0] *= 20; acts[..., 1] *= 2 * np.pi
    acts = acts.to(dtype)
    for k in range(10):
        env.step(acts[k % 8])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        env.step(acts[k % 8])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def time_rollout(n, dtype, sigma, K, reps=3):
    import torch
    from mr_rl_b200 import VecMREnv
    env = VecMREnv(n, device="cuda:0", dtype=dtype, noise="philox" if sigma else "none", seed=1, auto_reset=True)
    env.reset(init=None, noise_var=sigma, a0=1.0)
    env.rollout(policy="random", k_steps=K)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        env.rollout(policy="random", k_steps=K)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def measure(a):
    import torch
    tag = os.environ.get("MR_STEP_PATH", "default")
    # box calibration: plain device copy of the same footprint (63 MB read + 97 MB written ~ 80 MB copy)
    src = torch.empty(80 * 1024 * 1024, dtype=torch.uint8, device="cuda:0")
    dst = torch.empty_like(src)
    for _ in range(5):
        dst.copy_(src)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    cms = e0.elapsed_time(e1) / 50
    print(f"calibration: 160 MB copy traffic in {cms*1e3:.1f} us = {160*1.048576/cms:.0f} GB/s", flush=True)
    configs = [(torch.float64, 0.0, False), (torch.float64, 1.0, False), (torch.float32, 0.0, False),
               (torch.float32, 1.0, False), (torch.float64, 1.0, True)]
    for dtype, sigma, sp in configs:
        ms = time_step(a.n, dtype, sigma, a.steps, sp=sp)
        name = str(dtype)[6:]
        gbs = (BYTES[name] + (2 * dtype.itemsize if sp else 0)) * a.n / (ms * 1e-3) / 1e9
        print(f"step {name} sigma={sigma}{' state_prime' if sp else ''}: {ms*1e3:8.1f} us  vec={tag}  "
              f"{a.n/ms/1e6:8.2f} Genv-steps/s  {gbs:7.0f} GB/s algorithmic", flush=True)
    if a.rollout:
        for sigma in (0.0, 1.0):
            ms = time_rollout(a.n, torch.float64, sigma, 64)
            print(f"rollout K=64 float64 sigma={sigma}: {ms*1e3:8.1f} us  {a.n*64/ms/1e6:8.2f} Genv-steps/s", flush=True)


LINE = re.compile(r"^((?:step|rollout) [^:]+): +([0-9.]+) us")


def run_child(lib, argv):
    env = dict(os.environ, MR_LIB_PATH=os.path.abspath(lib))
    r = subprocess.run([sys.executable, *argv], cwd=ROOT, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{' '.join(argv)} with {lib} failed:\n{r.stdout}\n{r.stderr}")
    return r.stdout


def ab(a):
    if len(a.ab) < 2:
        sys.exit("--ab needs two or more libraries")
    libs = {chr(ord("A") + k): lib for k, lib in enumerate(a.ab)}
    for tag, lib in libs.items():
        if not os.path.exists(lib):
            sys.exit(f"{tag}: no library at {lib}")
        print(f"{tag} = {lib}", flush=True)
    child = [os.path.abspath(__file__), "--n", str(a.n), "--steps", str(a.steps)] + (["--rollout"] if a.rollout else [])
    bench = [os.path.join(ROOT, "bench.py"), "--no-extras", "--cpu-seconds", "1"]
    res = {tag: {} for tag in libs}
    order = list(libs)
    for rnd in range(a.rounds):
        for tag in order if rnd % 2 == 0 else order[::-1]:
            out = run_child(libs[tag], child)
            for line in out.splitlines():
                m = LINE.match(line)
                if m:
                    res[tag].setdefault(m.group(1), []).append(float(m.group(2)))
            if a.bench:
                last = [ln for ln in run_child(libs[tag], bench).splitlines() if ln.startswith("{")][-1]
                d = json.loads(last)
                res[tag].setdefault("bench.py headline (us per step)", []).append(d["ms_per_step"] * 1e3)
                res[tag].setdefault("bench.py headline value (Genv-steps/s)", []).append(d["value"] / 1e9)
            print(f"round {rnd} {tag}: " + ", ".join(f"{k} {v[-1]:.2f}" for k, v in res[tag].items()), flush=True)
    print(f"\n{'configuration':40s} " + " ".join(f"{t + ' median [min-max]':>24s} {t + '/A':>6s}" for t in libs), flush=True)
    for key in res["A"]:
        ma = statistics.median(res["A"][key])
        cols = []
        for tag in libs:
            v = res[tag].get(key, [])
            m = statistics.median(v)
            cols.append(f"{f'{m:.2f} [{min(v):.2f}-{max(v):.2f}]':>24s} {m / ma:6.4f}")
        print(f"{key:40s} " + " ".join(cols), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rollout", action="store_true")
    ap.add_argument("--ab", nargs="+", metavar="LIB", help="compare two or more library builds, alternating")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--bench", action="store_true", help="with --ab: add the bench.py headline to every round")
    a = ap.parse_args()
    if a.ab:
        ab(a)
    else:
        measure(a)
