"""bench.py — env-steps/s of the batched MR_Env hot path on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference's CPU path (port)
    python bench.py --dump-outputs DIR ...                          # + the last timed step's obs, rew, done as DIR/*.npy

A "step" is ONE launch of the single-step kernel (MR_Env.step for every env of the rank) on
synthetic random actions: fp64 storage, sigma = 1 (MR_Env.reset default) drawn by the in-kernel
Philox generator, auto reset on done.  BASELINE configs[2] as written: 2^20 envs in total, env i on
rank i // (2^20 / N), no data-path collective (strong scaling, the default; NCCL only sums the
episode statistics).  At N > 1 a rank's launch is a few microseconds of L2-resident work, so the K
timed launches run as one CUDA-graph replay; the weak-scaling curve (2^20 envs per GPU) is measured
in the same run and reported under "weak_scaling_1M_envs_per_gpu".
`value` is whole-job env-steps/s with inputs resident in HBM; `e2e` is the same metric through the
host-buffer call (host actions in, numpy obs/rew/done out, copies inside the timed region).
Timing: W warm-up launches, then the same kernel back to back for 0.1 s (untimed pre-roll), then ev0
directly behind the last pre-roll launch, exactly K launches, ev1.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
BYTES_PER_ENV_STEP = {"f64": 153, "f32": 81}     # SURVEY.md §8(d): algorithmic bytes, single-step path
PREROLL_S = 0.1     # the timed kernel runs back to back this long (untimed) right before ev0: clocks ramped, caches warm
# With --dump-outputs the pre-roll is this many launches instead (0.06 s at 2^20 fp64 envs, B200 at 1000 W): the env
# state carries over from step to step, so the dumped step must have the same number of steps before it in every run.
DUMP_PREROLL_LAUNCHES = 2048
DUMP_BUDGET_BYTES = 60 << 20      # array bytes: with the .npy headers a dump stays under 64 MB, even of 10^6 bytes


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs in total (strong scaling) / per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default, BASELINE configs[2] as written): --envs envs sharded over the ranks; "
                         "weak: --envs envs per GPU")
    ap.add_argument("--launch", default="auto", choices=["auto", "graph", "direct"],
                    help="the K timed single-step launches as one CUDA graph replay or as K stream launches "
                         "(auto: graph when a rank holds fewer than 2^20 envs)")
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--sigma", type=float, default=1.0)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--preroll-s", type=float, default=PREROLL_S,
                    help="seconds of the timed kernel run back to back right before the timed region (shrink it for an ncu pass)")
    ap.add_argument("--no-extras", action="store_true", help="skip the fused-rollout / small-batch side numbers")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (obs, rew, done of every env) as DIR/<name>.npy; "
                         "the pre-roll then has a fixed length, so the same arguments give the same arrays in every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ---- clocks during the timed region -----------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if (t0 is None or t >= t0 - 0.05) and (t1 is None or t <= t1 + 0.15)] or \
               [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except Exception:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "MEASURED_PEAKS.json hbm_gbs (measured)"
    except Exception:
        return {"hbm_gbs": 6650.0}, "B200_PROFILING.md fallback 6.65 TB/s"


# ---- CPU legs -----------------------------------------------------------------------------------
def cpu_port_throughput(budget_s, sigma):
    """The reference's numpy/scipy env restated on the real scipy RK45 (oracle/scipy_env.py), one
    process per host core, bounded sample.  Returns (value, cores, sample description, extras)."""
    from oracle import scipy_env
    cores = os.cpu_count() or 1
    probe = scipy_env.throughput(1, 4, 50, sigma)                       # ~0.05 s calibration
    per_core = max(probe["steps_per_s"], 1.0)
    steps = 100
    envs_per_proc = int(max(4, min(512, budget_s * per_core / steps)))
    r = scipy_env.throughput(cores, envs_per_proc, steps, sigma)
    sample = f"{cores} procs x {envs_per_proc} envs x {steps} steps, random actions, sigma={sigma}, auto reset"
    return r["steps_per_s"], cores, sample, {"single_core_steps_per_s": per_core}


def c_port_throughput(sigma):
    try:
        from oracle import c_oracle
        r = c_oracle.throughput(1 << 16, 32, sigma)
        return {"value": r["steps_per_s"], "unit": UNIT, "threads": r["threads"],
                "sample": "plain-C oracle, 65536 envs x 32 steps"}
    except Exception as e:   # no compiler on the box etc.
        return {"unavailable": str(e)[:120]}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (Python + scipy RK45; the
    reference sources cannot travel, so this is the oracle port pinned to them) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import scipy_env
    cores = os.cpu_count() or 1
    probe = scipy_env.throughput(1, 4, 50, args.sigma)
    total = args.steps + args.warmup
    envs_per_proc = int(max(2, min(256, 90.0 * probe["steps_per_s"] / max(total, 1))))
    scipy_env.throughput(cores, envs_per_proc, max(args.warmup, 1), args.sigma)           # warm-up pass
    t0 = time.perf_counter()
    r = scipy_env.throughput(cores, envs_per_proc, args.steps, args.sigma)
    wall = time.perf_counter() - t0
    sample_envs = cores * envs_per_proc
    value = r["steps_per_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * r["busy_s"] / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "1M batched MR_Env, single-step path (configs[2]), random actions (bounded CPU sample)",
                   "sample_envs": sample_envs, "sigma": args.sigma, "a0": 1.0, "auto_reset": True},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{cores} procs x {envs_per_proc} envs x {args.steps} steps (oracle/scipy_env.py on scipy RK45)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(line), file=_OUT, flush=True)


# ---- this repo's arm ---------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from mr_rl_b200 import VecMREnv

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def all_ranks(v):
        if world > 1:
            t = torch.zeros(world, dtype=torch.float64, device=dev)
            t[rank] = v
            dist.all_reduce(t)
            return [float(x) for x in t.tolist()]
        return [v]

    def gather_rows(t):
        """[n, ...] rows of every rank, in env order, as one numpy array on rank 0 (None elsewhere)."""
        t = t.contiguous()
        if world == 1:
            return t.cpu().numpy()
        sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([t.shape[0]], dtype=torch.int64, device=dev))
        m = max(int(s) for s in sizes)
        padded = torch.zeros((m, *t.shape[1:]), dtype=t.dtype, device=dev)
        padded[:t.shape[0]] = t
        parts = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(parts, padded)
        return torch.cat([p[:int(s)] for p, s in zip(parts, sizes)]).cpu().numpy() if rank == 0 else None

    strong = args.scaling == "strong"
    n_total = args.envs
    from mr_rl_b200 import shard_range
    if strong:
        base, n = shard_range(n_total, rank, world)          # env i lives on rank i // (n_total / world) (SURVEY 8e)
    else:
        base, n = rank * n_total, n_total
    tdt = torch.float64 if args.dtype == "f64" else torch.float32
    noise = "philox" if args.sigma != 0 else "none"
    pool = 8
    K = args.steps
    W = max(args.warmup, 3)

    def make_actions(m, seed):
        gen = torch.Generator(device=dev).manual_seed(seed)
        a = torch.rand(pool, m, 2, generator=gen, device=dev, dtype=torch.float64)
        a[..., 0] *= 20.0
        a[..., 1] *= 2 * np.pi
        return a.to(tdt)

    def make_env(m, env_base, sigma=args.sigma, kind=None, **kw):
        e = VecMREnv(m, device=dev, dtype=tdt, noise=kind or ("philox" if sigma != 0 else "none"), seed=2024,
                     env_base=env_base, auto_reset=True, **kw)
        e.want_state_prime = False                           # the 153 B/env-step accounting has no state_prime row
        e.reset(init=None, noise_var=sigma, a0=1.0)
        return e

    def timed_steps(e, a, steps, use_graph, preroll_s=None):
        """W warm-up steps, then the SAME kernel back to back for >= preroll_s (still untimed: the clocks ramp and
        settle under load), then — with no synchronisation or idle gap after the last pre-roll launch — ev0, exactly
        `steps` single-step launches, ev1.  use_graph: the K launches are one CUDA-graph replay (captured once; the
        pre-roll replays the same graph).  Returns (ms of the K steps, wall-clock window from the start of the pre-roll,
        pre-roll launches, ms of the pre-roll, graph, what the last step returned)."""
        preroll_s = args.preroll_s if preroll_s is None else preroll_s
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g = e.capture_steps([a[k] for k in range(pool)], steps) if use_graph else None
        p0.record()
        for k in range(W):
            e.step(a[k % pool])
        p1.record()
        torch.cuda.synchronize()
        per = max(p0.elapsed_time(p1) / W, 1e-3)              # ms per launch, rough (cold)
        n_pre = DUMP_PREROLL_LAUNCHES if args.dump_outputs else int(min(20000, max(8, preroll_s * 1e3 / per)))
        barrier()
        t_pre = time.perf_counter()
        p0.record()
        if g is not None:
            n_pre = max(2, n_pre // steps) * steps            # whole replays of the K-step graph
            for _ in range(n_pre // steps):
                g.replay()
            t0 = time.perf_counter()
            e0.record()
            out = g.replay()
            e1.record()
        else:
            for k in range(n_pre):
                e.step(a[k % pool])
            t0 = time.perf_counter()
            e0.record()
            for k in range(steps):
                out = e.step(a[k % pool])
            e1.record()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        barrier()
        return e0.elapsed_time(e1), (t_pre, t1), n_pre, p0.elapsed_time(e0), g, out

    # ---- headline: BASELINE configs[2] as written — `envs` envs sharded over the ranks, single-step path ---------------
    use_graph = args.launch == "graph" or (args.launch == "auto" and n < (1 << 20))
    env = make_env(n, base)
    acts = make_actions(n, 1234 + rank)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_local, (t_wall0, t_wall1), n_pre, ms_pre, graph, last = timed_steps(env, acts, K, use_graph)
    if args.dump_outputs:                                     # the next launch overwrites these buffers: copy them now
        last = {"obs": gather_rows(last[0]), "rew": gather_rows(last[1]), "done": gather_rows(last[2])}
    per_rank_ms = all_ranks(ms_local / K)
    ms = max_over_ranks(ms_local)
    launches = K + (1 if use_graph else 0)                   # kernels inside the timed region (graph: + the counter kernel)
    # consistency: three more windows of K steps each, directly after (GPU still warm) — the spread is reported
    repeats = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if graph is not None:
            graph.replay()
        else:
            for k in range(K):
                env.step(acts[k % pool])
        e1.record()
        torch.cuda.synchronize()
        repeats.append(e0.elapsed_time(e1) / K)
    # the timed region lasts a few ms — shorter than nvidia-smi's sampling period — so the same kernel
    # keeps running (untimed) for ~0.4 s while the clock sampler collects its under-load samples
    if rank == 0:
        t_ext = time.perf_counter()
        while time.perf_counter() - t_ext < 0.4:
            if graph is not None:
                graph.replay()
            else:
                for k in range(50):
                    env.step(acts[k % pool])
            torch.cuda.synchronize()
        t_wall1 = time.perf_counter()
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if clocks is not None:
        clocks["window"] = ("%.3f s pre-roll (%d launches) + timed region + 0.4 s of the same kernel back to back "
                            "(20 ms nvidia-smi period)" % (ms_pre * 1e-3, n_pre))
    barrier()
    env.check_status()

    envs_all = n_total if strong else world * n_total
    value = envs_all * K / (ms * 1e-3)
    ms_per_step = ms / K

    # ---- roofline of the dominant (only) kernel: CUDA-event time per launch ------------------
    peaks, peak_src = measured_peaks()
    bytes_per_launch = BYTES_PER_ENV_STEP[args.dtype] * n
    achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": None, "kernel": "env_step_tma_kernel",
                "algorithmic_bytes_per_env_step": BYTES_PER_ENV_STEP[args.dtype], "peak_source": peak_src,
                "frac_of_nominal_8TBs": achieved / 8000.0,
                "note": None if n * BYTES_PER_ENV_STEP[args.dtype] > 126e6 else
                        "this rank's working set (%.0f MB) is L2-resident: the launch is latency-bound, the HBM roofline "
                        "does not bound it" % (bytes_per_launch / 1e6)}
    prof = os.path.join(ROOT, "profiles", "traffic_step_kernel.json")
    if os.path.exists(prof):
        try:
            with open(prof) as f:
                tr = json.load(f)
            roofline["traffic"] = tr.get(args.dtype + ("_philox" if args.sigma else "_none")) if n == (1 << 20) else None
            roofline["traffic_source"] = tr.get("source", "ncu --set full capture of this kernel at 2^20 envs, profiles/")
        except Exception:
            pass

    # ---- e2e: host buffers through the public call, copies inside the timed region -----------------
    el = 8 if args.dtype == "f64" else 4

    def time_host(e, host_inputs, steps):
        t_pre = time.perf_counter()
        k = 0
        while k < 3 or time.perf_counter() - t_pre < 0.06:          # >= 60 ms of the same call before the timed region
            e.step_host(host_inputs[k % len(host_inputs)]); k += 1
        barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            e.step_host(host_inputs[k % len(host_inputs)])
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    e2e_steps = max(3, args.e2e_steps)
    host_acts = [acts[k % pool].cpu().pin_memory() for k in range(min(pool, e2e_steps))]   # pinned host inputs
    e2e_local = time_host(env, host_acts, e2e_steps)
    e2e_rank_ms = all_ranks(e2e_local / e2e_steps)
    e2e_ms = max_over_ranks(e2e_local)
    # bytes per step over the host link: actions in; obs rows x, y, d and the done byte out (the goal rows are the
    # constant 0 and the reward the constant 10 of MR_env.py:57,89 — written once on the host, never transferred)
    e2e = {"value": envs_all * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": n * 2 * el,
           "d2h_bytes_per_step": n * (3 * el + 1), "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
           "per_rank_ms_per_step": e2e_rank_ms,
           "api": "VecMREnv.step_host(pinned host actions) -> numpy obs, rew, done (float64 on the wire)"}
    e2e_extra = {}
    try:
        np_acts = [a.numpy().copy() for a in host_acts]             # plain (pageable) numpy arrays: + one copy into pinned memory
        ms_np = max_over_ranks(time_host(env, np_acts, e2e_steps))
        e2e_extra["e2e_numpy_unpinned_input"] = {"value": envs_all * e2e_steps / (ms_np * 1e-3), "unit": UNIT,
                                                 "ms_per_step": ms_np / e2e_steps}
        if args.dtype == "f64":
            env.host_io_dtype = torch.float32                       # float32 on the wire, fp64 state (the 1e-4 tier)
            f32_acts = [a.float().pin_memory() for a in host_acts]
            ms_32 = max_over_ranks(time_host(env, f32_acts, e2e_steps))
            env.host_io_dtype = None
            e2e_extra["e2e_float32_wire"] = {"value": envs_all * e2e_steps / (ms_32 * 1e-3), "unit": UNIT,
                                             "ms_per_step": ms_32 / e2e_steps, "h2d_bytes_per_step": n * 8,
                                             "d2h_bytes_per_step": n * 13}
    except Exception as ex:
        e2e_extra["e2e_extra_error"] = str(ex)[:160]

    # ---- episode statistics: the path's only collective -----------------------------------------------
    env.reset_stats()
    env.rollout(policy="random", k_steps=64)            # > one episode (51 steps) for every env
    stats = env.allreduce_stats()

    extras = dict(e2e_extra)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def side(name, fn):
        """A side number never breaks the headline."""
        try:
            fn()
        except Exception as ex:
            extras[name] = {"error": str(ex)[:200]}

    # ---- the other scaling curve + the same launches without a graph ------------------------------------
    if world > 1 and not args.no_extras:
        def weak():
            ew = make_env(1 << 20, rank * (1 << 20))
            aw = make_actions(1 << 20, 99 + rank)
            msw = timed_steps(ew, aw, K, False)[0]
            msw = max_over_ranks(msw) / K
            extras["weak_scaling_1M_envs_per_gpu"] = {
                "value": world * (1 << 20) / (msw * 1e-3), "unit": UNIT, "ms_per_step": msw, "envs_total": world << 20,
                "roofline_frac": BYTES_PER_ENV_STEP[args.dtype] * (1 << 20) / (msw * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "limit": "none: independent ranks, HBM-bound kernel at full size"}
        side("weak_scaling_1M_envs_per_gpu", weak)
    if use_graph and not args.no_extras:
        def direct():
            msd = timed_steps(env, acts, K, False)[0]
            msd = max_over_ranks(msd) / K
            extras["same_steps_without_cuda_graph"] = {"value": envs_all / (msd * 1e-3), "unit": UNIT, "ms_per_step": msd}
        side("same_steps_without_cuda_graph", direct)

    if not args.no_extras and args.sigma != 0.0:
        # the same single-step kernel with sigma = 0 (MR_simulator.py:18 default noise_var): no RNG work
        def noise_free():
            env0 = make_env(n, base, sigma=0.0)
            ms0_local = timed_steps(env0, acts, K, use_graph)[0]
            ms0 = max_over_ranks(ms0_local) / K
            ach0 = bytes_per_launch / (ms0 * 1e-3) / 1e9
            extras["noise_free_sigma0"] = {"value": envs_all / (ms0 * 1e-3), "unit": UNIT, "ms_per_step": ms0,
                                           "roofline": {"bound": "hbm", "achieved": ach0, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                                        "frac": ach0 / peaks["hbm_gbs"]}}
        side("noise_free_sigma0", noise_free)
    if not args.no_extras:
        def with_sp():
            env.want_state_prime = True
            mss = timed_steps(env, acts, K, False)[0]
            env.want_state_prime = False
            mss = max_over_ranks(mss) / K
            b = (BYTES_PER_ENV_STEP[args.dtype] + 2 * el) * n
            extras["with_state_prime_rows"] = {"value": envs_all / (mss * 1e-3), "unit": UNIT, "ms_per_step": mss,
                                               "bytes_per_env_step": BYTES_PER_ENV_STEP[args.dtype] + 2 * el,
                                               "roofline_frac": b / (mss * 1e-3) / 1e9 / peaks["hbm_gbs"]}
        side("with_state_prime_rows", with_sp)

        # fused K = 64 rollout on the same envs (state in registers; FP64-pipe bound)
        def fused():
            env.rollout(policy="random", k_steps=64)
            barrier()
            ev0.record()
            reps = 3
            for _ in range(reps):
                env.rollout(policy="random", k_steps=64)
            ev1.record()
            torch.cuda.synchronize()
            fms = max_over_ranks(ev0.elapsed_time(ev1)) / reps
            extras["fused_rollout_k64"] = {"value": envs_all * 64 / (fms * 1e-3), "unit": UNIT, "ms_per_launch": fms,
                                           "envs_per_gpu": n, "actions": "in-kernel Philox", "sigma": args.sigma}
        side("fused_rollout_k64", fused)
    if not args.no_extras and rank == 0 and world == 1:
        side_numbers_rank0(args, extras, dev, tdt, noise, peaks, el)
    barrier()

    if rank == 0:
        if world == 1:
            cpu_val, cores, sample, cpu_extra = cpu_port_throughput(args.cpu_seconds, args.sigma)
            cpu_baseline = {"value": cpu_val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                            "implementation": "oracle/scipy_env.py: reference env restated on scipy.integrate.RK45",
                            **cpu_extra, "c_port": c_port_throughput(args.sigma)}
        else:
            cpu_baseline = {"skipped": "the CPU baseline is timed on rank 0 at N=1 only"}
        limit = ("HBM bandwidth (one launch moves %.0f MB per GPU)" % (bytes_per_launch / 1e6)) if bytes_per_launch > 126e6 else \
                ("per-launch latency: %.0f MB per rank is L2-resident and one launch is only %.1f us of work; "
                 "the K launches run as one CUDA graph with programmatic dependent launch between them" % (bytes_per_launch / 1e6, ms_per_step * 1e3))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": "1M batched MR_Env sharded over the GPUs, single-step path (configs[2]), random actions",
                       "envs_total": envs_all, "envs_per_gpu": n, "sigma": args.sigma, "a0": 1.0,
                       "noise": "in-kernel Philox4x32-7 + Box-Muller" if args.sigma else "none (sigma=0)",
                       "auto_reset": True, "sharding": f"env i on rank i // {n}, {world} rank(s), no data-path collective",
                       "launch": "CUDA graph of the K single-step launches" if use_graph else "K stream launches",
                       "limited_by": limit,
                       "l2_policy": "state+outputs per step = %.0f MB %s 126 MB L2; 8 rotating action buffers"
                                    % (bytes_per_launch / 1e6, ">" if bytes_per_launch > 126e6 else "<")},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": launches,
            "clocks": clocks, "repeat_ms_per_step": repeats, "per_rank_ms_per_step": per_rank_ms, "preroll_launches": n_pre,
            "episode_stats_allreduced": stats, **extras,
        }
        if args.dump_outputs:
            line["dumped_outputs"] = write_outputs(args.dump_outputs, last)
        print(json.dumps(line), file=_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def write_outputs(dirname, arrays):
    """Write each [n, ...] array as dirname/<name>.npy, float64 kept and anything else as float32.  If the set is larger
    than DUMP_BUDGET_BYTES, every array keeps the same fixed, seeded sample of rows, whose indices go to env_index.npy.
    Returns {name: shape}."""
    import numpy as np
    arrays = {k: v.astype(v.dtype if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v[:1].nbytes for v in arrays.values())
    if n * row_bytes > DUMP_BUDGET_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BUDGET_BYTES // (row_bytes + 8), replace=False))
        arrays = {"env_index": rows.astype(np.float64), **{k: v[rows] for k, v in arrays.items()}}
    os.makedirs(dirname, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), np.ascontiguousarray(v))
    return {k: list(v.shape) for k, v in arrays.items()}


def _static_traffic(key):
    """DRAM bytes per launch from the committed ncu capture (profiles/traffic_step_kernel.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic_step_kernel.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


def side_numbers_rank0(args, extras, dev, tdt, noise, peaks, el):
    """BASELINE configs[1], [3], [4], the parity-mode roofline and the SURVEY 8f rows — one GPU, rank 0."""
    import numpy as np
    import torch

    from mr_rl_b200 import VecMREnv
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 1 << 20

    def side(name, fn):
        try:
            fn()
        except Exception as ex:
            extras[name] = {"error": str(ex)[:200]}

    # ---- parity mode (BASELINE.md 4 row 2): table-driven noise, 281 B per env-step in fp64 ----------------------
    def parity_mode():
        steps_per_cycle, K = 48, min(args.steps, 40)
        L = 4 + 16 * steps_per_cycle
        gen = torch.Generator(device=dev).manual_seed(7)
        table = torch.randn(L, n, generator=gen, device=dev, dtype=torch.float64)       # 6.5 GB, shared by all cycles
        e = VecMREnv(n, device=dev, dtype=tdt, noise="table", noise_table=table, auto_reset=False)
        e.want_state_prime = False
        a = torch.rand(8, n, 2, generator=gen, device=dev, dtype=torch.float64)
        a[..., 0] *= 20.0
        a[..., 1] *= 2 * np.pi
        a = a.to(tdt)
        t_pre = time.perf_counter()
        while time.perf_counter() - t_pre < 0.15:                   # untimed cycles: reset (rewinds the cursors) + 48 steps
            e.reset(init=None, noise_var=1.0, a0=1.0)
            for k in range(steps_per_cycle):
                e.step(a[k % 8])
            torch.cuda.synchronize()
        e.reset(init=None, noise_var=1.0, a0=1.0)
        for k in range(steps_per_cycle - K):
            e.step(a[k % 8])
        ev0.record()
        for k in range(K):
            e.step(a[k % 8])
        ev1.record()
        torch.cuda.synchronize()
        e.check_status()
        ms = ev0.elapsed_time(ev1) / K
        b = (BYTES_PER_ENV_STEP[args.dtype] + 128) * n
        assert int(e._cursor[:n].min()) == int(e._cursor[:n].max()) == L      # 16 draws per step, every env
        extras["parity_mode_table_noise"] = {
            "value": n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "kernel": "env_step_tma_kernel<table> (noise rows bulk-copied per tile)",
            "roofline": {"bound": "hbm", "achieved": b / (ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": b / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         "algorithmic_bytes_per_env_step": BYTES_PER_ENV_STEP[args.dtype] + 128,
                         "traffic": _static_traffic(args.dtype + "_table")}}
        del e, table
    side("parity_mode_table_noise", parity_mode)

    # BASELINE configs[1]: 4096 envs, fused K = 64
    def config1():
        small = VecMREnv(4096, device=dev, dtype=tdt, noise=noise, seed=5, auto_reset=True)
        small.reset(init=None, noise_var=args.sigma, a0=1.0)
        for _ in range(200):
            small.rollout(policy="random", k_steps=64)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(50):
            small.rollout(policy="random", k_steps=64)
        ev1.record()
        torch.cuda.synchronize()
        sms = ev0.elapsed_time(ev1) / 50
        extras["config1_4096_envs_k64"] = {"value": 4096 * 64 / (sms * 1e-3), "unit": UNIT, "ms_per_launch": sms}
    side("config1_4096_envs_k64", config1)

    # BASELINE configs[4]: DDPG actor (MR_ddpg architecture, random init) driving 2^20 envs for 1000 steps
    def config4():
        from mr_rl_b200 import init_actor, pack_actor
        env = VecMREnv(n, device=dev, dtype=tdt, noise=noise, seed=11, auto_reset=True)
        env.reset(init=None, noise_var=args.sigma, a0=1.0)
        packed = pack_actor(init_actor(0), dev)
        env.rollout(policy=packed, k_steps=50)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(20):                                          # 20 launches x 50 fused steps = 1000 steps
            env.rollout(policy=packed, k_steps=50)
        ev1.record()
        torch.cuda.synchronize()
        ams = ev0.elapsed_time(ev1)
        env.check_status()
        # BASELINE.md 3.3: torch-CPU fp32 forward of the same MLP on the box's host cores (a reported baseline)
        from mr_rl_b200.actor import torch_reference
        params = init_actor(0)
        obs_cpu = np.zeros((65536, 5), np.float32)
        obs_cpu[:, :2] = np.random.default_rng(0).uniform(100, 120, (65536, 2))
        obs_cpu[:, 4] = np.hypot(obs_cpu[:, 0], obs_cpu[:, 1])
        torch_reference(params, obs_cpu)
        t0 = time.perf_counter()
        for _ in range(5):
            torch_reference(params, obs_cpu)
        t_cpu = (time.perf_counter() - t0) / 5
        extras["config4_actor_in_loop_1000_steps"] = {
            "cpu_torch_actor_forwards_per_s": 65536 / t_cpu, "cpu_threads": torch.get_num_threads(),
            "value": n * 1000 / (ams * 1e-3), "unit": UNIT, "ms_total": ams, "envs": n, "steps": 1000, "launches": 20,
            "actor": "5-64-BN-ReLU-64-BN-ReLU-2 tanh, fp32 accuracy; both dense layers on tcgen05 (3xFP16 passes, TMEM accumulators), "
                     "persistent CTAs, 4 per SM"}
    side("config4_actor_in_loop_1000_steps", config4)

    # BASELINE configs[3]: GP disturbance model, 2000 training points, 262144 queries (both GPs, mean + std)
    def config3():
        from mr_rl_b200 import DeviceGP
        rng = np.random.default_rng(0)
        X = np.sort(rng.uniform(-np.pi, np.pi, 2000))
        yx = 0.2 + 0.5 * np.cos(X + 0.3) + 0.09 * rng.standard_normal(2000)
        yy = -0.1 + 0.4 * np.sin(X - 0.2) + 0.09 * rng.standard_normal(2000)
        q = torch.rand(262144, device=dev, dtype=torch.float64) * 6.28 - 3.14
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gps = [DeviceGP.fit(X, yv, ls, 0.008, device=dev) for yv, ls in ((yx, 0.2), (yy, 0.25))]   # fixed kernels (SURVEY 8d C4)
        torch.cuda.synchronize()
        t_fit = (time.perf_counter() - t0) * 1e3

        def both(std):
            for g in gps:
                g.predict(q, std)
            torch.cuda.synchronize()
            ev0.record()
            for g in gps:
                g.predict(q, std)
            ev1.record()
            torch.cuda.synchronize()
            return ev0.elapsed_time(ev1)
        tri = both(True)                                             # sklearn's algorithm: |L^-1 k|^2, triangular DMMA kernel
        mean_only = both(False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        proj_rows = [g.enable_spectral_variance() for g in gps]      # low-rank form, verified against the triangular one
        torch.cuda.synchronize()
        t_spec_build = (time.perf_counter() - t0) * 1e3
        spec = both(True)
        # BASELINE.md 3.2: sklearn's GPR.predict on the box's host cores, 4096 of the queries (it is linear in the query count)
        from sklearn.gaussian_process import GaussianProcessRegressor
        from sklearn.gaussian_process.kernels import RBF, WhiteKernel
        gpr = GaussianProcessRegressor(kernel=RBF(0.2) + WhiteKernel(0.008), optimizer=None, alpha=1e-10).fit(X[:, None], yx)
        qs = q[:4096].cpu().numpy()[:, None]
        gpr.predict(qs[:256], return_std=True)
        t0 = time.perf_counter()
        gpr.predict(qs, return_std=True)
        t_sk_std = time.perf_counter() - t0
        t0 = time.perf_counter()
        gpr.predict(qs)
        t_sk_mean = time.perf_counter() - t0
        extras["config3_gp_262k_queries_2k_train"] = {
            "cpu_sklearn": {"sample": "GaussianProcessRegressor.predict, one GP, 4096 queries x 2000 training points, default BLAS threads",
                            "cores": os.cpu_count(), "mean_std_queries_per_s_per_gp": 4096 / t_sk_std,
                            "mean_only_queries_per_s_per_gp": 4096 / t_sk_mean},
            "reference_algorithm_triangular_ms_both_gps": tri, "spectral_ms_both_gps": spec, "mean_only_ms_both_gps": mean_only,
            "queries_per_s_triangular": 262144 / (tri * 1e-3), "queries_per_s_spectral": 262144 / (spec * 1e-3),
            "triangular_tflops_fp64": 2 * (262144 * 2048.0 * 2048 / 2 * 2) / (tri * 1e-3) / 1e12,
            "model_fit_ms_both_gps": t_fit,
            "spectral_model_build_ms_both_gps": t_spec_build,
            "spectral_model_build": "one-time set-up outside the timed predict: eigendecomposition of the 2048^2 Gram matrix "
                                    "(torch.linalg.eigh = cuSOLVER, LIBRARY) + a 512-query check against the triangular form",
            "variance_projection_rows": proj_rows,
            "kernels": "triangular: gp_kq_mean_kernel + gp_var_kernel (fp64 DMMA m8n8k4, lower-triangular right operand); "
                       "spectral: gp_posterior_spectral_kernel (mean + std fused, verified to 1e-9 or refused)"}
    side("config3_gp_262k_queries_2k_train", config3)

    # SURVEY 8f rows: the GPR fit with sklearn's 5-restart search driven from the host, the DDPG learner
    def next_rows():
        from mr_rl_b200 import DDPGLearner, DeviceGPR, LearningModule, OUNoise, ReplayBuffer
        from mr_rl_b200.ddpg import train as _train
        rng = np.random.default_rng(1)
        Xf = np.sort(rng.uniform(-np.pi, np.pi, size=(1970, 1)), axis=0)
        yf = 0.8 * np.sin(2 * Xf[:, 0]) + 0.3 * np.cos(Xf[:, 0]) + 0.15 * rng.standard_normal(1970)
        DeviceGPR(n_restarts_optimizer=0, random_state=3, device=dev).fit(Xf[:256], yf[:256])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gpr = DeviceGPR(n_restarts_optimizer=5, random_state=3, device=dev).fit(Xf, yf)
        torch.cuda.synchronize()
        t_fit = time.perf_counter() - t0
        rb = ReplayBuffer(10000, 0, device=dev)
        env_t = VecMREnv(4096, device=dev, noise="philox", seed=0, auto_reset=True)
        learner, ou = DDPGLearner(device=dev), OUNoise(4096, device=dev)
        _train(env_t, learner, ou, min_batch=64, steps=20, replay=rb)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _train(env_t, learner, ou, min_batch=64, steps=200, replay=rb)
        torch.cuda.synchronize()
        t_it = (time.perf_counter() - t0) / 200
        ev0.record()
        for _ in range(50):
            learner.update(rb, 64)
        ev1.record()
        torch.cuda.synchronize()
        t_upd = ev0.elapsed_time(ev1) / 50 * 1e3
        # LearningModule.predict for 262144 desired velocities (SURVEY 8f rank 1) on the config-3 GPs
        lm = LearningModule(device=dev)
        g1 = DeviceGPR(optimizer=None, length_scale=0.2, noise_level=0.008, device=dev).fit(Xf, yf)
        g2 = DeviceGPR(optimizer=None, length_scale=0.25, noise_level=0.008, device=dev).fit(Xf, 0.5 * yf)
        lm.set_models(g1, g2, 1.5, 4.0, 0.2, -0.1)
        ang = torch.rand(262144, device=dev, dtype=torch.float64) * 6.28 - 3.14
        vdes = 6.0 * torch.stack([torch.cos(ang), torch.sin(ang)], 1)
        lm.predict_batch(vdes)
        torch.cuda.synchronize()
        ev0.record()
        lm.predict_batch(vdes)
        ev1.record()
        torch.cuda.synchronize()
        t_head = ev0.elapsed_time(ev1)
        extras["next_rows"] = {
            "lm_predict_batch_262k_ms": t_head,     # heading search + posterior (mean, std of both GPs) at the minimiser
            "corrected_headings_path": "Chebyshev interpolants of the GP means (verified)" if lm._cheb is not None else "direct kernel sums",
            "gpr_search_n1970_5_restarts_s": t_fit, "gpr_objective_evals": gpr.n_objective_evals,
            "gpr_theta": [float(v) for v in gpr.kernel_.theta],
            "ddpg_update_batch64_us": t_upd,
            "ddpg_train_iteration_4096_envs_ms": t_it * 1e3,
            "note": "mr_gp_fit per objective evaluation; one mr_ddpg_update launch per learner update"}
    side("next_rows", next_rows)


def _claim_stdout():
    """Only the JSON line may reach stdout: libraries (e.g. NCCL's version banner) write to fd 1 too, so
    fd 1 is pointed at stderr for the run and the saved descriptor is used for the final line."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, "w")


if __name__ == "__main__":
    a = parse()
    _OUT = _claim_stdout()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
