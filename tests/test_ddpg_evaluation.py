"""Greedy evaluation of DDPG populations and population-based training (evaluate_population, evaluate, pbt_plan,
pbt_population, DDPGPopulation.exploit / set_hyper / hyper_table; mr_ddpg_evaluate_population).

Without a GPU: the C struct layout, every argument error of the entry point, the Python-level ValueErrors and pbt_plan.
On the GPU, every member's rows against a solo env that resets at the evaluation's step index and runs the plain actor
rollout: lengths and outcomes exact, returns bit for bit (fp64 storage), statistics equal to the reduction of the rows;
then CTAs that change member, early exit, common random numbers, the memory the launch does not own, and PBT."""
import ctypes as C
import math
import os
import subprocess
import types

import numpy as np
import pytest
import torch

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "mr_rl_b200.h")
FAKE = C.c_void_p(256)          # a non-null address that no argument check dereferences


def test_eval_struct_matches_c_layout(tmp_path):
    from mr_rl_b200 import _lib as L
    prog = tmp_path / "ev.c"
    fields = [f[0] for f in L.DDPGEval._fields_]
    body = "\n".join(f'printf("{f} %zu\\n", offsetof(mr_ddpg_eval, {f}));' for f in fields)
    prog.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "{HEADER}"\nint main(void){{{body}\n'
                    'printf("size %zu\\n", sizeof(mr_ddpg_eval));return 0;}\n')
    exe = tmp_path / "ev"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert C.sizeof(L.DDPGEval) == int(out["size"])
    for f in fields:
        assert getattr(L.DDPGEval, f).offset == int(out[f]), f


def _eval_args():
    from mr_rl_b200 import _lib as L
    ev = L.DDPGEval(FAKE, 3, 1, 256, None, FAKE, FAKE, FAKE, FAKE, FAKE, 0)
    p = L.default_params()
    nz = L.Noise(L.NOISE_PHILOX, 0, None, 0, 1, 0, 0, None)
    tt = L.TimeTable(FAKE, 64, 0)
    return ev, p, nz, tt


def _call(ev, p, nz, tt, dtype=0):
    from mr_rl_b200 import _lib as L
    lib = L.load()
    rc = lib.mr_ddpg_evaluate_population(C.byref(ev) if ev is not None else None, dtype, C.byref(p) if p is not None else None,
                                         C.byref(nz) if nz is not None else None, C.byref(tt) if tt is not None else None, None)
    return rc, lib.mr_last_error().decode()


def test_evaluate_population_argument_errors_need_no_gpu():
    from mr_rl_b200 import _lib as L
    ev, p, nz, tt = _eval_args()
    fn = "mr_ddpg_evaluate_population"
    for args in ((None, p, nz, tt), (ev, None, nz, tt), (ev, p, None, tt)):
        rc, msg = _call(*args)
        assert rc == -1 and f"{fn}: null evaluation, params or noise" in msg
    bad = L.DDPGEval.from_buffer_copy(ev)
    bad.actors = None
    rc, msg = _call(bad, p, nz, tt)
    assert rc == -1 and "null actor" in msg
    for m in (0, -1, 257):
        bad = L.DDPGEval.from_buffer_copy(ev)
        bad.members = m
        rc, msg = _call(bad, p, nz, tt)
        assert rc == -1 and "members must be in 1..256" in msg, m
    for n in (0, -128, 100, 129, 1 << 30):
        bad = L.DDPGEval.from_buffer_copy(ev)
        bad.member_envs = n
        rc, msg = _call(bad, p, nz, tt)
        assert rc == -1 and "member_envs must be a positive multiple of 128" in msg, n
    rc, msg = _call(ev, p, nz, tt, dtype=7)
    assert rc == -1 and "bad dtype" in msg
    for length in (0, 1, 50):                        # K = max_timesteps + 1 = 51
        rc, msg = _call(ev, p, nz, L.TimeTable(FAKE, length, 0))
        assert rc == -1 and "at least max_timesteps + 1 = 51" in msg, length
    rc, msg = _call(ev, p, nz, L.TimeTable(None, 64, 0))
    assert rc == -1 and "time table" in msg
    p2 = L.SimParams.from_buffer_copy(p)
    p2.max_timesteps = -1
    rc, msg = _call(ev, p2, nz, tt)
    assert rc == -1 and "max_timesteps" in msg
    p2 = L.SimParams.from_buffer_copy(p)
    p2.time_span = 0.0
    rc, msg = _call(ev, p2, nz, tt)
    assert rc == -1 and "time_span" in msg
    nz2 = L.Noise.from_buffer_copy(nz)
    nz2.offset_dev = FAKE.value
    rc, msg = _call(ev, p, nz2, tt)
    assert rc == -1 and "offset_dev" in msg
    nz2 = L.Noise.from_buffer_copy(nz)
    nz2.mode = 9
    rc, msg = _call(ev, p, nz2, tt)
    assert rc == -1 and "unknown noise mode" in msg
    nz2 = L.Noise.from_buffer_copy(nz)
    nz2.mode = L.NOISE_NONE                          # default noise_var = 1
    rc, msg = _call(ev, p, nz2, tt)
    assert rc == -1 and "needs a noise source" in msg
    # table noise: a table, then N columns with common random numbers, members x N without
    tab = L.Noise(L.NOISE_TABLE, 0, FAKE, 0, 1, 0, 0, None)
    rc, msg = _call(ev, p, tab, tt)
    assert rc == -1 and "table noise without a table" in msg
    tab.table_len = 100
    for crn, cols, ok in ((1, 255, False), (1, 256, True), (0, 256, False), (0, 767, False), (0, 768, True)):
        e2 = L.DDPGEval.from_buffer_copy(ev)
        e2.common_random_numbers, e2.table_cols = crn, cols
        old = L.set_actor_path("simt")               # every check passes -> the actor path check answers last
        try:
            rc, msg = _call(e2, p, tab, tt)
        finally:
            L.set_actor_path(old)
        if ok:
            assert rc == -3 and "CUDA-core actor path" in msg, (crn, cols)
        else:
            assert rc == -1 and f"has {cols} columns, the evaluation reads" in msg, (crn, cols)
    old = L.set_actor_path("simt")
    try:
        rc, msg = _call(ev, p, nz, tt)
        assert rc == -3 and "CUDA-core actor path" in msg
    finally:
        L.set_actor_path(old)


def _cpu_env(**kw):
    from mr_rl_b200 import _lib as L
    env = types.SimpleNamespace(params=L.default_params(), per_env_params=False, device=torch.device("cpu"),
                                dtype=torch.float64, noise_kind="philox")
    env.params.reward_mode = L.REWARD_SHAPED
    env.__dict__.update(kw)
    return env


def test_evaluation_python_value_errors_need_no_gpu():
    from mr_rl_b200 import _lib as L
    from mr_rl_b200.ddpg import evaluate, evaluate_population, pbt_population
    count = L.load().mr_actor_param_count()
    pop = types.SimpleNamespace(members=3, actor=torch.zeros(3, count), action_bound=(20.0, 2 * math.pi))
    env = _cpu_env()
    for m in (0, 257):
        with pytest.raises(ValueError, match="members must be in 1..256"):
            evaluate_population(env, types.SimpleNamespace(members=m, actor=pop.actor, action_bound=pop.action_bound), 128)
    for n in (0, -128, 100, 200):
        with pytest.raises(ValueError, match="must be a positive multiple of 128"):
            evaluate_population(env, pop, n)
    with pytest.raises(ValueError, match="action_bound must equal"):
        evaluate_population(env, types.SimpleNamespace(members=3, actor=pop.actor, action_bound=(10.0, 1.0)), 128)
    with pytest.raises(ValueError, match="per-env parameter rows"):
        evaluate_population(_cpu_env(per_env_params=True), pop, 128)
    with pytest.raises(ValueError, match=f"the actors must be \\[3, {count}\\]"):
        evaluate_population(env, types.SimpleNamespace(members=3, actor=torch.zeros(2, count), action_bound=pop.action_bound), 128)
    for init in (torch.zeros(127, 2), torch.zeros(128, 3), torch.zeros(3)):
        with pytest.raises(ValueError, match="init must be \\(2,\\) or \\(128, 2\\)"):
            evaluate_population(env, pop, 128, init=init)
    tab = _cpu_env(noise_kind="table", _noise_table=torch.zeros(10, 256))
    with pytest.raises(ValueError, match="the noise table has 256 columns; the evaluation reads 384"):
        evaluate_population(tab, pop, 128, common_random_numbers=False)
    with pytest.raises(ValueError, match="the noise table has 256 columns; the evaluation reads 384"):
        evaluate_population(tab, pop, 384)
    learner = types.SimpleNamespace(actor=torch.zeros(count), action_bound=pop.action_bound)
    with pytest.raises(ValueError, match="must be a positive multiple of 128"):
        evaluate(env, learner, 1000)
    const = _cpu_env()
    const.params.reward_mode = L.REWARD_CONST10
    with pytest.raises(ValueError, match="constant reward"):
        pbt_population(const, pop, None, None, 2, 64, 128)
    for r, s in ((0, 64), (2, 0)):
        with pytest.raises(ValueError, match="rounds and steps_per_round must be at least 1"):
            pbt_population(env, pop, None, None, r, s, 128)


def test_pbt_plan():
    from mr_rl_b200.ddpg import pbt_plan
    rng = np.random.default_rng(3)
    scores = rng.normal(size=16)
    a, b = pbt_plan(scores, 0.25, rng=7), pbt_plan(scores, 0.25, rng=7)
    for x, y in zip(a, b):                             # one seed, one plan
        assert np.array_equal(x, y)
    dst, src, factors = a
    order = np.argsort(-scores, kind="stable")
    assert list(dst) == list(order[12:])               # the bottom quarter, in ranking order
    assert set(src) <= set(order[:4])                  # copies a top-quarter member
    assert factors.shape == (4, 3) and set(np.unique(factors)) <= {0.8, 1.25}   # only copied members draw factors
    assert any(not np.array_equal(pbt_plan(scores, 0.25, rng=s)[1], src) for s in range(8, 20))   # src is drawn
    # ties rank by member index, lower first; NaN ranks last
    dst, src, _ = pbt_plan([1.0, 2.0, 2.0, 1.0, 0.5, 2.0], 1 / 3, rng=0)
    assert list(dst) == [3, 4] and set(src) <= {1, 2}
    dst, _, _ = pbt_plan([math.nan, 1.0, 2.0, 3.0], 0.25, rng=0)
    assert list(dst) == [0]
    # fraction 0: nothing is copied and nothing is drawn
    g = np.random.default_rng(5)
    dst, src, factors = pbt_plan(scores, 0.0, rng=g)
    assert dst.size == src.size == 0 and factors.shape == (0, 3)
    assert g.integers(0, 2**62) == np.random.default_rng(5).integers(0, 2**62)
    # fraction 0.5: the bottom half copies from the top half, every member of one half
    dst, src, factors = pbt_plan(scores, 0.5, perturb=(0.5, 2.0), rng=1)
    assert sorted(dst) == sorted(order[8:]) and set(src) <= set(order[:8]) and set(np.unique(factors)) <= {0.5, 2.0}
    assert factors.shape == (8, 3)
    for f in (-0.1, 0.51, 1.0):
        with pytest.raises(ValueError, match="fraction must be in \\[0, 0.5\\]"):
            pbt_plan(scores, f)


# ---------------------------------------------------------------------------------------------------------------------
# GPU

DEV = "cuda:0"
SENTINEL = 77
BOUND, MAX_T, TABLE_LEN = 60.0, 30, 16384   # the solo runs step on after the terminal step: a table that lasts


def _task(env, dtype_np=np.float64):
    """Start positions and bounds that end episodes every way: at the goal on the first step, out of bounds, and by
    timeout, with tiles that mix the three."""
    from mr_rl_b200 import Box
    env.max_timesteps = MAX_T
    env.observation_space = Box(low=np.array([-BOUND, -BOUND, -BOUND, -BOUND, 0]), high=np.array([BOUND, BOUND, BOUND, BOUND, 80000]))
    env.init_space = Box(low=np.array([-65.0, -65.0]), high=np.array([65.0, 65.0]))


def _starts(N, seed=2):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(N, 2, generator=g, dtype=torch.float64) * 130 - 65).to(DEV)


def _population(P, seed=8):
    from mr_rl_b200.ddpg import DDPGPopulation
    pop = DDPGPopulation(P, seeds=[3 * p + 1 for p in range(P)], device=DEV)
    g = torch.Generator(device=DEV).manual_seed(seed)
    pop.actor.add_(0.05 * torch.randn(pop.actor.shape, generator=g, device=DEV))   # actions off the tanh's flat part
    return pop


class Case:
    """An evaluation env and, per member, the solo env whose rows the member's must equal."""

    def __init__(self, P, N, dtype=torch.float64, noise="philox", reward="shaped", mism=False, crn=True, sigma=1.0, seed=5):
        from mr_rl_b200 import VecMREnv
        self.P, self.N, self.crn, self.mism, self.sigma = P, N, crn, mism, sigma
        self.kw = dict(device=DEV, dtype=dtype, noise=noise, seed=seed, reward_mode=reward)
        self.table = None
        width = N if crn else P * N
        if noise == "table":
            self.table = torch.randn(TABLE_LEN, width, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
        self.env = VecMREnv(width, noise_table=self.table, auto_reset=True, **self.kw)
        _task(self.env)
        self.env.reset(noise_var=sigma, a0=1.0, is_mismatched=mism)

    def solo(self, p, actor, init, offset):
        """Member p's solo run: reset at step index ``offset`` (previous model flag = the evaluated one), then the plain
        actor rollout of K steps, recorded."""
        from mr_rl_b200 import VecMREnv
        N = self.N
        base = 0 if self.crn else p * N
        tab = None if self.table is None else (self.table if self.crn else self.table[:, p * N:(p + 1) * N])
        se = VecMREnv(N, env_base=base, noise_table=tab, auto_reset=False, **self.kw)
        _task(se)
        se.params.is_mismatched = 1 if self.mism else 0
        se._step_index = offset
        se.reset(init=init, noise_var=self.sigma, a0=1.0, is_mismatched=self.mism)
        res = se.rollout(policy=actor, k_steps=MAX_T + 1, record_episodes=True)
        return se, res


def _solo_rows(se, res, dtype):
    """length, outcome, return (sequential float64 sum through the first terminal step) and status of a solo run."""
    done = res["done_traj"].cpu().numpy().astype(bool)
    assert done.any(0).all()                         # every episode ends within K steps
    t = done.argmax(0)
    n = done.shape[1]
    step = res["step"].cpu().numpy()
    length = step[t, np.arange(n)]
    xy = res["xy"].cpu().numpy().astype(np.float64)
    x, y = xy[t, 0, np.arange(n)], xy[t, 1, np.arange(n)]
    inside = (np.abs(x) <= BOUND) & (np.abs(y) <= BOUND)
    outcome = np.where(~inside, 2, np.where(length > MAX_T, 3, 1))
    rew = res["rew_traj"].cpu().numpy().astype(np.float64)
    ret = np.array([np.add.accumulate(rew[:t[j] + 1, j])[-1] for j in range(n)])
    return length, outcome, ret, se.status.cpu().numpy()


def _assert_member_equals_solo(res, p, solo_rows, dtype):
    length, outcome, ret, status = solo_rows
    assert np.array_equal(res.length[p].cpu().numpy(), length), p
    assert np.array_equal(res.outcome[p].cpu().numpy(), outcome), p
    assert np.array_equal(res.status[p].cpu().numpy(), status), p
    got = res.ret[p].cpu().numpy()
    if dtype is torch.float64:
        assert np.array_equal(got, ret), p
    else:                                            # the solo's recorded rewards are float32 (-0.1f)
        assert np.abs(got - ret).max() <= 1e-6 * (MAX_T + 1), p


def _assert_stats_reduce_rows(res, stats, N):
    for p in range(res.ret.shape[0]):
        length, outcome = res.length[p].double(), res.outcome[p]
        st = stats[p].cpu().numpy()
        want = {0: N, 1: float(length.sum()), 3: float((outcome == 1).sum()), 4: float((outcome == 2).sum()),
                5: float((outcome == 3).sum()), 6: float(length.sum()), 7: float((res.status[p] != 0).sum())}
        for k, v in want.items():
            assert st[k] == v, (p, k)
        r = float(res.ret[p].sum())
        assert abs(st[2] - r) <= 1e-12 * max(1.0, abs(r)), p


def _evaluate_with_stats(case, pop, init, offset):
    """evaluate_population, and the statistics rows of the same evaluation from the C entry point (the Python result
    keeps rates)."""
    from mr_rl_b200 import _lib as L
    from mr_rl_b200.ddpg import evaluate_population
    P, N, e = pop.members, case.N, case.env
    res = evaluate_population(e, pop, N, init=init, common_random_numbers=case.crn, offset=offset, per_env=True)
    stats = torch.zeros(P, L.STATS_LEN, dtype=torch.float64, device=DEV)
    init_t = init.to(e.dtype).contiguous() if init is not None else None
    ev = L.DDPGEval(pop.actor.data_ptr(), P, 1 if case.crn else 0, N, init_t.data_ptr() if init_t is not None else None,
                    stats.data_ptr(), None, None, None, None, case.table.shape[1] if case.table is not None else 0)
    nz = L.Noise.from_buffer_copy(e._noise_for(e.params.noise_var))
    nz.offset = offset
    L.check(L.load().mr_ddpg_evaluate_population(C.byref(ev), e._dt, C.byref(e.params), C.byref(nz), C.byref(e._c_tt), None))
    torch.cuda.synchronize()
    return res, stats


@pytest.mark.gpu
@pytest.mark.parametrize("N", [128, 256])
@pytest.mark.parametrize("path", ["tf32", "default"])
@pytest.mark.parametrize("crn", [True, False])
@pytest.mark.parametrize("mism", [False, True])
@pytest.mark.parametrize("reward", ["shaped", "const"])
@pytest.mark.parametrize("noise", ["philox", "none", "table"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_evaluation_equals_solo_runs(dtype, noise, reward, mism, crn, path, N):
    from mr_rl_b200 import _lib as L
    P, offset = 3, 1234
    old = L.set_actor_path(path)
    try:
        case = Case(P, N, dtype, noise, reward, mism, crn, sigma=0.0 if noise == "none" else 1.0)
        pop = _population(P)
        init = _starts(N) if N == 128 else None          # N = 256: the starts are samples of init_space
        res, stats = _evaluate_with_stats(case, pop, init, offset)
        solos = [case.solo(p, pop.actor[p], init, offset) for p in range(P)]
        torch.cuda.synchronize()
    finally:
        L.set_actor_path(old)
    for p, (se, r) in enumerate(solos):
        _assert_member_equals_solo(res, p, _solo_rows(se, r, dtype), dtype)
    _assert_stats_reduce_rows(res, stats, N)
    out = res.outcome.cpu().numpy()
    assert (out == 1).any() and (out == 3).any()       # episodes end at the goal and by timeout
    assert torch.equal(res.env_steps.cpu(), res.length.sum(1).double().cpu())


@pytest.mark.gpu
def test_evaluation_many_members_per_cta():
    """More tiles than resident 3xFP16 CTAs (640 > 4 x 148): persistent CTAs restage weights and flush statistics rows
    when they move on to another member."""
    P, N = 5, 128 * 128
    case = Case(P, N, crn=False)
    pop = _population(P)
    init = _starts(N, seed=3)
    res, stats = _evaluate_with_stats(case, pop, init, 77)
    for p in range(P):
        se, r = case.solo(p, pop.actor[p], init, 77)
        _assert_member_equals_solo(res, p, _solo_rows(se, r, torch.float64), torch.float64)
    _assert_stats_reduce_rows(res, stats, N)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["tf32", "default"])
def test_early_exit_is_invisible(path):
    """Tiles whose envs mix starts inside the goal (done after one step) with starts that time out: the rows equal the
    solo runs', which step every env K times."""
    from mr_rl_b200 import _lib as L
    P, N = 2, 256
    init = _starts(N, seed=4)
    init[::2] = 1.0                                   # inside min_dist2goal: the goal on the first step
    init[256 - 128:] = 0.5                            # the second tile ends entirely after one step
    init[1:128:2] = torch.tensor([40.0, 40.0], dtype=torch.float64, device=DEV)
    old = L.set_actor_path(path)
    try:
        case = Case(P, N, sigma=0.0, noise="none")
        pop = _population(P)
        res, stats = _evaluate_with_stats(case, pop, init, 5)
        for p in range(P):
            se, r = case.solo(p, pop.actor[p], init, 5)
            _assert_member_equals_solo(res, p, _solo_rows(se, r, torch.float64), torch.float64)
    finally:
        L.set_actor_path(old)
    ln = res.length.cpu().numpy()
    assert (ln[:, ::2] == 1).all() and (ln[:, 128:] == 1).all() and (ln[:, 1:128:2] > 1).all()
    assert (stats[:, 5] > 0).all().item()             # timeouts beside the one-step episodes


@pytest.mark.gpu
def test_common_random_numbers():
    from mr_rl_b200.ddpg import evaluate, evaluate_population
    P, N = 2, 256
    case = Case(P, N, crn=True)
    big = Case(P, N, crn=False)
    pop = _population(P)
    pop.actor[1].copy_(pop.actor[0])
    for c, crn in ((case, True), (big, False)):
        res = evaluate_population(c.env, pop, N, common_random_numbers=crn, offset=3, per_env=True)
        same = all(torch.equal(getattr(res, f)[0], getattr(res, f)[1]) for f in ("ret", "length", "outcome", "status"))
        assert same == crn, crn
    # a different offset draws other starts and noise
    a = evaluate_population(case.env, pop, N, offset=3, per_env=True)
    b = evaluate_population(case.env, pop, N, offset=4, per_env=True)
    assert not torch.equal(a.ret, b.ret)
    # one learner: member 1's rows (with common random numbers every member draws what env j draws)
    one = evaluate(case.env, pop.member(1), N, offset=3, per_env=True)
    for f in ("ret", "length", "outcome", "status"):
        assert torch.equal(getattr(one, f)[0], getattr(a, f)[1]), f


@pytest.mark.gpu
def test_evaluation_writes_nothing_else():
    """Sentinels around the statistics and per-env rows; the env passed in stays bit for bit as it was."""
    from mr_rl_b200 import _lib as L
    from mr_rl_b200.ddpg import evaluate_population
    P, N, pad = 3, 128, 40
    case = Case(P, N, dtype=torch.float32, noise="table", crn=False)
    pop = _population(P)
    e = case.env
    e.rollout(policy="random", k_steps=3)               # a state that is not the reset one
    before = {k: getattr(e, k).clone() for k in ("_state", "_counter", "_cursor", "_status", "_obs", "_rew", "_done", "_sp",
                                                  "_stats")}
    step_index = e._step_index
    stats = torch.full((P + 2, 8), float(SENTINEL), dtype=torch.float64, device=DEV)
    stats[1:P + 1] = 0
    rows = {n: torch.full((P * N + 2 * pad,), SENTINEL, dtype=dt, device=DEV)
            for n, dt in (("ret", torch.float64), ("length", torch.int32), ("outcome", torch.uint8), ("status", torch.uint8))}
    ev = L.DDPGEval(pop.actor.data_ptr(), P, 0, N, None, stats[1].data_ptr(),
                    *[rows[n][pad:].data_ptr() for n in ("ret", "length", "outcome", "status")], case.table.shape[1])
    nz = L.Noise.from_buffer_copy(e._noise_for(e.params.noise_var))
    nz.offset = 9
    L.check(L.load().mr_ddpg_evaluate_population(C.byref(ev), e._dt, C.byref(e.params), C.byref(nz), C.byref(e._c_tt), None))
    res = evaluate_population(e, pop, N, common_random_numbers=False, offset=9, per_env=True)
    torch.cuda.synchronize()
    assert (stats[0] == SENTINEL).all() and (stats[P + 1] == SENTINEL).all() and (stats[1:P + 1, 0] == N).all()
    for n, t in rows.items():
        assert (t[:pad] == SENTINEL).all() and (t[pad + P * N:] == SENTINEL).all(), n
        assert torch.equal(t[pad:pad + P * N].view(P, N), getattr(res, n)), n
    assert (rows["outcome"][pad:pad + P * N] != SENTINEL).all()
    for k, v in before.items():
        assert torch.equal(getattr(e, k), v), k
    assert e._step_index == step_index


@pytest.mark.gpu
def test_exploit_and_hyper():
    P = 5
    pop = _population(P)
    pop.set_hyper(3, actor_lr=2e-3, critic_lr=3e-2, tau=5e-3, gamma=0.9)
    for p in range(P):
        g = torch.Generator(device=DEV).manual_seed(p)
        for t in pop._moments:
            t[p].copy_(torch.rand(t.shape[1], generator=g, device=DEV))
    tensors = lambda: [pop.actor, pop.actor_target, pop.critic, pop.critic_target, *pop._moments]
    before = [t.clone() for t in tensors()]
    h_before = pop.hyper_table()
    pop.exploit([0, 4], [3, 1])
    for t, b in zip(tensors(), before):
        assert torch.equal(t[0], b[3]) and torch.equal(t[4], b[1])
        for p in (1, 2, 3):
            assert torch.equal(t[p], b[p])
    h = pop.hyper_table()
    assert np.array_equal(h[0], h_before[3]) and np.array_equal(h[4], h_before[1])
    assert np.array_equal(h[1:4], h_before[1:4])
    assert tuple(h[0]) == (2e-3, 3e-2, 5e-3, 0.9)
    for p in range(P):                                # the member learners see the same rows and storage
        m = pop.member(p)
        assert (m.hyper.lr_actor, m.hyper.lr_critic, m.hyper.tau, m.hyper.gamma) == tuple(h[p])
        assert m.actor.data_ptr() == pop.actor[p].data_ptr()
    pop.exploit([1, 2], [2, 1])                       # a swap: every source is read before a destination is written
    assert torch.equal(pop.actor[1], before[0][2]) and torch.equal(pop.actor[2], before[0][1])
    with pytest.raises(ValueError, match="dst repeats a member"):
        pop.exploit([1, 1], [2, 3])
    with pytest.raises(ValueError, match="member 5 is not in 0..4"):
        pop.exploit([5], [0])
    with pytest.raises(ValueError, match="tau must be finite"):
        pop.set_hyper(0, tau=math.nan)


def _pbt_setup(P=4, N=128, seed=0):
    from mr_rl_b200 import VecMREnv
    from mr_rl_b200.ddpg import DDPGPopulation, OUNoise, PopulationReplay
    env = VecMREnv(P * N, device=DEV, noise="philox", seed=seed, auto_reset=True, reward_mode="shaped")
    env.max_timesteps = 20
    pop = DDPGPopulation(P, seeds=list(range(P)), actor_lr=[1e-3, 2e-3, 5e-4, 1e-3], critic_lr=1e-2, device=DEV)
    return env, pop, OUNoise(P * N, device=DEV), PopulationReplay(P, 4096, 0, device=DEV)


@pytest.mark.gpu
def test_pbt_with_nothing_copied_equals_plain_training():
    """fraction = 0: the evaluations between the rounds leave training untouched."""
    from mr_rl_b200 import _lib as L
    from mr_rl_b200.ddpg import pbt_population, train_population
    old = L.set_actor_path("tf32")
    try:
        env, pop, noise, rep = _pbt_setup()
        hist = pbt_population(env, pop, noise, rep, rounds=3, steps_per_round=16, eval_envs=128, fraction=0.0, collect_steps=8)
        env2, pop2, noise2, rep2 = _pbt_setup()
        train_population(env2, pop2, noise2, replay=rep2, steps=48, collect_steps=8)
        torch.cuda.synchronize()
    finally:
        L.set_actor_path(old)
    for a, b in zip([pop.actor, pop.critic, pop.actor_target, pop.critic_target, *pop._moments],
                    [pop2.actor, pop2.critic, pop2.actor_target, pop2.critic_target, *pop2._moments]):
        assert torch.equal(a, b)
    assert torch.equal(env._state, env2._state) and torch.equal(rep.s, rep2.s) and torch.equal(noise.x_prev, noise2.x_prev)
    assert hist["score"].shape == (3, 4) and hist["hyper"].shape == (3, 4, 4)
    assert (hist["parent"] == np.arange(4)).all()


@pytest.mark.gpu
def test_pbt_is_deterministic():
    from mr_rl_b200.ddpg import pbt_population
    runs = []
    for _ in range(2):
        env, pop, noise, rep = _pbt_setup()
        hist = pbt_population(env, pop, noise, rep, rounds=3, steps_per_round=16, eval_envs=128, fraction=0.25, seed=11,
                              collect_steps=8)
        torch.cuda.synchronize()
        runs.append((hist, pop.actor.clone(), pop.hyper_table()))
    (h1, a1, t1), (h2, a2, t2) = runs
    for k in ("score", "hyper", "parent"):
        assert np.array_equal(h1[k], h2[k]), k
    assert torch.equal(a1, a2) and np.array_equal(t1, t2)
    assert (h1["parent"] != np.arange(4)).any()        # one member per round was replaced
    assert np.isfinite(h1["score"]).all()
