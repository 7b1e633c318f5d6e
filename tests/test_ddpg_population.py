"""DDPG populations (DDPGPopulation, PopulationReplay, collect_population, train_population; mr_ddpg_update_population,
mr_env_rollout_ddpg_collect_population).

Without a GPU: the C struct layout, every argument error of both entry points and the Python-level ValueErrors.  On the
GPU, every check is bit for bit against the solo runs of the members: the population update against mr_ddpg_update, one
collect launch against each member's solo collect (3xTF32 and 3xFP16 actor paths, fp64 and fp32 storage, through auto
resets and a ring that wraps), train_population against solo train(collect_steps=K), and the memory neither launch owns."""
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


def test_population_struct_matches_c_layout(tmp_path):
    from mr_rl_b200 import _lib as L
    prog = tmp_path / "pop.c"
    fields = [f[0] for f in L.DDPGPopulation._fields_]
    body = "\n".join(f'printf("{f} %zu\\n", offsetof(mr_ddpg_population, {f}));' for f in fields)
    prog.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "{HEADER}"\nint main(void){{{body}\n'
                    'printf("size %zu\\n", sizeof(mr_ddpg_population));\n'
                    'printf("max %d\\n", MR_DDPG_MAX_MEMBERS);return 0;}\n')
    exe = tmp_path / "pop"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert C.sizeof(L.DDPGPopulation) == int(out["size"])
    assert L.DDPG_MAX_MEMBERS == int(out["max"])
    for f in fields:
        assert getattr(L.DDPGPopulation, f).offset == int(out[f]), f


def _hyper(L, members):
    return (L.DDPGHyper * members)(*[L.DDPGHyper(0.99, 1e-3, 1e-3, 1e-2, (C.c_double * 2)(20.0, 6.28), 0.9, 0.999, 1e-8)
                                     for _ in range(members)])


def _update(pop, count=100, batch=64, update_index=1):
    from mr_rl_b200 import _lib as L
    lib = L.load()
    rc = lib.mr_ddpg_update_population(C.byref(pop) if pop is not None else None, count, batch, update_index, None, None)
    return rc, lib.mr_last_error().decode()


def test_update_population_argument_errors_need_no_gpu():
    from mr_rl_b200 import _lib as L
    P = 3
    hyper, seeds = _hyper(L, P), (C.c_uint64 * P)(1, 2, 3)
    pop = L.DDPGPopulation(P, L.DDPGState(*([FAKE] * 10)), L.Replay(FAKE, FAKE, FAKE, FAKE, FAKE, 128), hyper, seeds)
    fn = "mr_ddpg_update_population"
    rc, msg = _update(None)
    assert rc == -1 and f"{fn}: null population" in msg
    for m in (0, -1, 257):
        bad = L.DDPGPopulation.from_buffer_copy(pop)
        bad.members = m
        rc, msg = _update(bad)
        assert rc == -1 and "members must be in 1..256" in msg, m
    for field, _ in L.DDPGState._fields_:
        bad = L.DDPGPopulation.from_buffer_copy(pop)
        setattr(bad.st, field, None)
        rc, msg = _update(bad)
        assert rc == -1 and "null learner state" in msg, field
    for field in ("s", "a", "r", "d", "s2"):
        bad = L.DDPGPopulation.from_buffer_copy(pop)
        setattr(bad.ring, field, None)
        rc, msg = _update(bad)
        assert rc == -1 and "null replay ring array" in msg, field
    bad = L.DDPGPopulation.from_buffer_copy(pop)
    bad.hyper = None
    rc, msg = _update(bad)
    assert rc == -1 and "null hyper-parameters" in msg
    bad = L.DDPGPopulation.from_buffer_copy(pop)
    bad.seeds = None
    rc, msg = _update(bad)
    assert rc == -1 and "null seeds" in msg
    for b in (0, -3, 4097):
        rc, msg = _update(pop, count=5000, batch=b)
        assert rc == -1 and "batch must be in 1..4096" in msg, b
    for count in (63, 129):
        rc, msg = _update(pop, count=count)
        assert rc == -1 and "batch <= count <= capacity" in msg, count
    for u in (0, -1):
        rc, msg = _update(pop, update_index=u)
        assert rc == -1 and "update_index" in msg, u
    for field in ("gamma", "tau", "lr_actor", "lr_critic", "adam_beta1", "adam_beta2", "adam_eps"):
        for v in (math.nan, math.inf):
            h = _hyper(L, P)
            setattr(h[2], field, v)
            bad = L.DDPGPopulation(P, pop.st, pop.ring, h, seeds)
            rc, msg = _update(bad)
            assert rc == -1 and "hyper-parameters of member 2 must be finite" in msg, field
    h = _hyper(L, P)
    h[1].action_bound[1] = -math.inf
    rc, msg = _update(L.DDPGPopulation(P, pop.st, pop.ring, h, seeds))
    assert rc == -1 and "member 1 must be finite" in msg


def _collect_args():
    from mr_rl_b200 import _lib as L
    st = L.EnvState(*([FAKE] * 8), None, None, None)
    p = L.default_params()
    nz = L.Noise(L.NOISE_PHILOX, 0, None, 0, 1, 0, 0, None)
    tt = L.TimeTable(FAKE, 16, 0)
    io = L.RolloutIO()
    io.action_source, io.k_steps, io.actor = L.ACTIONS_ACTOR, 3, FAKE.value
    ring = L.Replay(FAKE, FAKE, FAKE, FAKE, FAKE, 300)
    c = L.DDPGCollect(FAKE, 0.15, 0.0, 0.3, 1e-2, 5, 0, 0, ring, 10)
    out = L.StepOut(FAKE, FAKE, FAKE, None, 1024, 0, 0)
    return st, p, nz, tt, io, c, out


def _collect(st, p, nz, tt, io, c, out, n=3 * 256, members=3, dtype=0):
    from mr_rl_b200 import _lib as L
    lib = L.load()
    rc = lib.mr_env_rollout_ddpg_collect_population(C.byref(st) if st is not None else None, n, dtype, C.byref(p), C.byref(nz),
                                                    C.byref(tt), C.byref(io) if io is not None else None,
                                                    C.byref(c) if c is not None else None, members,
                                                    C.byref(out) if out is not None else None, None)
    return rc, lib.mr_last_error().decode()


def test_collect_population_argument_errors_need_no_gpu():
    from mr_rl_b200 import _lib as L
    st, p, nz, tt, io, c, out = _collect_args()
    fn = "mr_env_rollout_ddpg_collect_population"
    for m in (0, -2, 257):
        rc, msg = _collect(st, p, nz, tt, io, c, out, members=m)
        assert rc == -1 and f"{fn}: members must be in 1..256" in msg, m
    for n, m in ((3 * 256 + 1, 3), (3 * 64, 3), (0, 3), (-256, 1), (384, 2), (256 * 5, 3)):
        rc, msg = _collect(st, p, nz, tt, io, c, out, n=n, members=m)
        assert rc == -1 and "n must be members x N with N a positive multiple of 128" in msg, (n, m)
    rc, msg = _collect(st, p, nz, tt, io, c, out, n=3 * 384)              # N = 384 > capacity 300
    assert rc == -1 and "N > capacity" in msg
    for head in (-1, 300, 1000):
        bad = L.DDPGCollect.from_buffer_copy(c)
        bad.head = head
        rc, msg = _collect(st, p, nz, tt, io, bad, out)
        assert rc == -1 and "0 <= head < capacity" in msg, head
    # the checks of the solo collector, with this entry point's name
    rc, msg = _collect(None, p, nz, tt, io, c, out)
    assert rc == -1 and f"{fn}: null state" in msg
    rc, msg = _collect(st, p, nz, tt, None, c, out)
    assert rc == -1 and "bad io" in msg
    io2 = L.RolloutIO.from_buffer_copy(io)
    io2.action_source = L.ACTIONS_PHILOX
    rc, msg = _collect(st, p, nz, tt, io2, c, out)
    assert rc == -1 and "must be MR_ACTIONS_ACTOR" in msg
    io2 = L.RolloutIO.from_buffer_copy(io)
    io2.actor = None
    rc, msg = _collect(st, p, nz, tt, io2, c, out)
    assert rc == -1 and "null actor" in msg
    rc, msg = _collect(st, p, nz, tt, io, None, out)
    assert rc == -1 and "null collect struct" in msg
    bad = L.DDPGCollect.from_buffer_copy(c)
    bad.ou_state = None
    rc, msg = _collect(st, p, nz, tt, io, bad, out)
    assert rc == -1 and "null ou_state" in msg
    for field in ("s", "a", "r", "d", "s2"):
        bad = L.DDPGCollect.from_buffer_copy(c)
        setattr(bad.ring, field, None)
        rc, msg = _collect(st, p, nz, tt, io, bad, out)
        assert rc == -1 and "null replay ring array" in msg, field
    rc, msg = _collect(st, p, nz, tt, io, c, None)
    assert rc == -1 and "out->obs" in msg
    bad = L.DDPGCollect.from_buffer_copy(c)
    bad.ring.capacity, bad.head = 0, 0
    rc, msg = _collect(st, p, nz, tt, io, bad, out)
    assert rc == -1 and "capacity must be positive" in msg
    for field in ("ou_theta", "ou_mu", "ou_sigma", "ou_dt"):
        bad = L.DDPGCollect.from_buffer_copy(c)
        setattr(bad, field, math.nan)
        rc, msg = _collect(st, p, nz, tt, io, bad, out)
        assert rc == -1 and "must be finite" in msg, field
    rc, msg = _collect(st, p, nz, L.TimeTable(None, 0, 0), io, c, out)
    assert rc == -1 and "time table" in msg
    st2 = L.EnvState.from_buffer_copy(st)
    st2.a0 = st2.noise_var = st2.is_mismatched = FAKE.value
    rc, msg = _collect(st2, p, nz, tt, io, c, out)
    assert rc == -3 and "per-env parameter rows" in msg
    old = L.set_actor_path("simt")
    try:
        rc, msg = _collect(st, p, nz, tt, io, c, out)
        assert rc == -3 and "CUDA-core actor path" in msg
    finally:
        L.set_actor_path(old)


def test_population_python_value_errors_need_no_gpu():
    from mr_rl_b200.ddpg import DDPGPopulation, PopulationReplay, collect_population, train_population
    for m in (0, 257):
        with pytest.raises(ValueError, match="members must be in 1..256"):
            DDPGPopulation(m)
        with pytest.raises(ValueError, match="members must be in 1..256"):
            PopulationReplay(m, 100)
    with pytest.raises(ValueError, match="seeds has 2 values for 3 members"):
        DDPGPopulation(3, seeds=[1, 2])
    for kw in ("actor_lr", "critic_lr", "tau", "gamma"):
        with pytest.raises(ValueError, match=f"{kw} has 4 values for 3 members"):
            DDPGPopulation(3, **{kw: [0.1] * 4})
    with pytest.raises(ValueError, match="random_seeds has 1 values for 2 members"):
        PopulationReplay(2, 100, random_seeds=[7])
    pop = types.SimpleNamespace(members=3, action_bound=(20.0, 2 * math.pi))
    rep = types.SimpleNamespace(members=3, buffer_size=1000)
    env = types.SimpleNamespace(num_envs=3 * 128)
    for n in (3 * 100, 3 * 128 + 3, 2 * 128):
        with pytest.raises(ValueError, match="must be members \\(3\\) x N with N a multiple of 128"):
            collect_population(types.SimpleNamespace(num_envs=n), pop, None, rep, 2)
    with pytest.raises(ValueError, match="k_steps must be at least 1"):
        collect_population(env, pop, None, rep, 0)
    with pytest.raises(ValueError, match="the replay has 2 members, the population 3"):
        collect_population(env, pop, None, types.SimpleNamespace(members=2, buffer_size=1000), 2)
    with pytest.raises(ValueError, match="replay buffer holds"):
        collect_population(env, pop, None, types.SimpleNamespace(members=3, buffer_size=100), 2)
    noise = types.SimpleNamespace(x_prev=torch.zeros(3 * 128 - 1, 2))
    with pytest.raises(ValueError, match="the OU noise has 383 processes for 384 envs"):
        collect_population(env, pop, noise, rep, 2)
    with pytest.raises(ValueError, match="collect_steps must be at least 1"):
        train_population(env, pop, None, collect_steps=0)
    with pytest.raises(ValueError, match="multiple of 128"):
        train_population(types.SimpleNamespace(num_envs=300), pop, None, collect_steps=4)
    with pytest.raises(ValueError, match="the replay has 4 members"):
        train_population(env, pop, None, collect_steps=4, replay=types.SimpleNamespace(members=4, buffer_size=1000))
    with pytest.raises(ValueError, match="the replay has 2 members"):
        DDPGPopulation.update(pop, types.SimpleNamespace(members=2), 64)
    for b in (0, 4097):
        with pytest.raises(ValueError, match="batch_size must be in 1..4096"):
            DDPGPopulation.update(pop, types.SimpleNamespace(members=3), b)


# ---------------------------------------------------------------------------------------------------------------------
# GPU

DEV = "cuda:0"
SENTINEL = 77.0
SEEDS = [0, 5, 9, 13, 21]
HYPER = dict(actor_lr=[1e-3, 3e-3, 1e-4, 2e-3, 5e-4], critic_lr=[1e-2, 3e-3, 2e-2, 1e-3, 5e-3],
             tau=[1e-3, 1e-2, 5e-3, 2e-3, 1e-3], gamma=[0.99, 0.9, 0.95, 0.99, 0.8])


def _hyper_of(P):
    return {k: v[:P] for k, v in HYPER.items()}


def _solo_learner(pop, p):
    """The solo learner member p was built as."""
    from mr_rl_b200.ddpg import DDPGLearner
    h = _hyper_of(pop.members)
    return DDPGLearner(actor_lr=h["actor_lr"][p], critic_lr=h["critic_lr"][p], tau=h["tau"][p], gamma=h["gamma"][p],
                       seed=pop.seeds[p], device=DEV)


def _learner_tensors(m):
    return [m.actor, m.actor_target, m.critic, m.critic_target, *m._moments]


def _fill_ring(rep, count, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    for t in (rep.s, rep.a, rep.s2):
        t.copy_(torch.randn(t.shape, generator=g, device=DEV) * 50)
    rep.r.copy_(torch.randn(rep.r.shape, generator=g, device=DEV))
    rep.d.copy_((torch.rand(rep.d.shape, generator=g, device=DEV) < 0.1).float())
    rep.count, rep.head = count, count % rep.buffer_size


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [64, 200])
def test_population_update_equals_solo_updates(batch):
    from mr_rl_b200 import _lib as L
    from mr_rl_b200.ddpg import DDPGPopulation, PopulationReplay
    P, cap, count = 5, 700, 650
    pop = DDPGPopulation(P, seeds=SEEDS, device=DEV, **_hyper_of(P))
    rep = PopulationReplay(P, cap, random_seeds=[3, 4, 5, 6, 7], device=DEV)
    _fill_ring(rep, count, 1)
    solos = [_solo_learner(pop, p) for p in range(P)]
    for p, m in enumerate(solos):                          # member p starts as its solo learner
        for a, b in zip(_learner_tensors(pop.member(p)), _learner_tensors(m)):
            assert torch.equal(a, b)
    rings = [rep.member(p) for p in range(P)]
    lib = L.load()
    infos = torch.zeros(P, 2, dtype=torch.float32, device=DEV)
    for u in range(1, 7):
        info = pop.update(rep, batch)
        for p, m in enumerate(solos):                      # the single-CTA kernel (no workspace) for every batch size
            rc = lib.mr_ddpg_update(C.byref(m._c), C.byref(rings[p]._c), count, batch, None, m.seed ^ rings[p].random_seed, u,
                                    C.byref(m.hyper), infos[p].data_ptr(), None, 0, None)
            L.check(rc, "mr_ddpg_update")
        torch.cuda.synchronize()
        assert torch.equal(info, infos), u
    assert pop.updates == 6
    for p, m in enumerate(solos):
        for a, b in zip(_learner_tensors(pop.member(p)) + pop.member(p)._grads, _learner_tensors(m) + m._grads):
            assert torch.equal(a, b), p
    assert len({float(pop.actor[p].sum()) for p in range(P)}) == P


class PopSetup:
    """members x N envs with a population and its OU noise and rings, plus each member's solo env, learner, noise and ring."""

    def __init__(self, P, N, dtype, capacity, head, reward_mode="shaped"):
        from mr_rl_b200 import VecMREnv
        from mr_rl_b200.ddpg import DDPGPopulation, OUNoise, PopulationReplay, ReplayBuffer
        self.P, self.N = P, N
        kw = dict(device=DEV, dtype=dtype, noise="philox", seed=3, auto_reset=True, reward_mode=reward_mode)
        self.env = VecMREnv(P * N, **kw)
        self.solo_envs = [VecMREnv(N, env_base=p * N, **kw) for p in range(P)]
        for e in (self.env, *self.solo_envs):
            e.max_timesteps = 5                            # episode boundaries inside the launch
            e.reset(noise_var=1.0, a0=1.0)
            e.reset_stats()
        self.pop = DDPGPopulation(P, seeds=SEEDS[:P], device=DEV, **_hyper_of(P))
        g = torch.Generator(device=DEV).manual_seed(8)
        self.pop.actor.add_(0.05 * torch.randn(self.pop.actor.shape, generator=g, device=DEV))   # actions off the tanh's flat part
        self.solos = [_solo_learner(self.pop, p) for p in range(P)]
        for p, m in enumerate(self.solos):
            m.actor.copy_(self.pop.actor[p])
        x0 = 0.2 * torch.randn(P * N, 2, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
        self.noise = OUNoise(P * N, sigma=0.3, seed=11, device=DEV)
        self.noise.x_prev.copy_(x0)
        self.noise.calls = 3                               # a process that has run before
        self.solo_noise = [OUNoise(N, sigma=0.3, seed=11, env_base=p * N, device=DEV) for p in range(P)]
        for p, nz in enumerate(self.solo_noise):
            nz.x_prev.copy_(x0[p * N:(p + 1) * N])
            nz.calls = 3
        self.rep = PopulationReplay(P, capacity, random_seeds=list(range(P)), device=DEV)
        self.solo_rb = [ReplayBuffer(capacity, p, device=DEV) for p in range(P)]
        for rb in (self.rep, *self.solo_rb):
            for t in (rb.s, rb.a, rb.r, rb.d, rb.s2):
                t.fill_(SENTINEL)
            rb.head, rb.count = head, head

    def collect(self, k, **kw):
        from mr_rl_b200.ddpg import collect, collect_population
        collect_population(self.env, self.pop, self.noise, self.rep, k, **kw)
        for p in range(self.P):
            collect(self.solo_envs[p], self.solos[p], self.solo_noise[p], self.solo_rb[p], k, **kw)

    def assert_equal_to_solo(self):
        P, N, e = self.P, self.N, self.env
        for p in range(P):
            sl, se = slice(p * N, (p + 1) * N), self.solo_envs[p]
            rb = self.solo_rb[p]
            for name in ("s", "a", "r", "d", "s2"):
                assert torch.equal(getattr(self.rep, name)[p], getattr(rb, name)), (p, name)
            assert torch.equal(self.noise.x_prev[sl], self.solo_noise[p].x_prev), p
            assert torch.equal(e._state[:, sl], se._state[:, :N]), p
            assert torch.equal(e._obs[:, sl], se._obs[:, :N]), p
            for a, b in ((e._counter, se._counter), (e._cursor, se._cursor), (e._status, se._status), (e._rew, se._rew),
                         (e._done, se._done)):
                assert torch.equal(a[sl], b[:N]), p
            got, want = self.pop.stats[p].cpu().numpy(), se.stats.cpu().numpy()
            for k in (0, 1, 3, 4, 5, 6, 7):                # integer statistics: exact
                assert got[k] == want[k], (p, k)
            assert abs(got[2] - want[2]) <= 1e-12 * abs(want[2]), p   # sum_reward: atomics add in any order
            assert (self.rep.head, self.rep.count, self.noise.calls) == (rb.head, rb.count, self.solo_noise[p].calls)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["tf32", "default"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("N", [256, 128])
def test_collect_population_equals_solo_collects(path, dtype, N):
    from mr_rl_b200 import _lib as L
    P, K = 3, 7
    cap = 5 * N + 17                                       # the first launch's K N > capacity: it wraps the ring
    old = L.set_actor_path(path)
    try:
        s = PopSetup(P, N, dtype, capacity=cap, head=cap - 40)
        s.collect(K)
        s.collect(3)
        torch.cuda.synchronize()
    finally:
        L.set_actor_path(old)
    s.assert_equal_to_solo()
    st = s.pop.stats.cpu().numpy()
    assert (st[:, 0] >= N).all()                           # every env crossed an episode boundary
    assert (st[:, 6] == 10 * N).all()
    assert not torch.equal(s.rep.a[0], s.rep.a[1]) and not torch.equal(s.rep.a[1], s.rep.a[2])   # each member its own actor
    assert s.rep.count == cap and s.rep.head == (cap - 40 + 10 * N) % cap


@pytest.mark.gpu
def test_collect_population_many_members_per_cta():
    """More tiles than resident 3xFP16 CTAs: persistent CTAs move from member to member (restaged weights, flushed
    statistics rows)."""
    P, N = 5, 128 * 128                                    # 640 tiles > 4 CTAs x 148 SMs
    s = PopSetup(P, N, torch.float64, capacity=2 * N, head=0)
    s.collect(2)
    torch.cuda.synchronize()
    s.assert_equal_to_solo()


@pytest.mark.gpu
def test_train_population_equals_solo_train():
    from mr_rl_b200 import VecMREnv, _lib as L
    from mr_rl_b200.ddpg import DDPGPopulation, OUNoise, ReplayBuffer, train, train_population
    P, N, K, steps = 3, 128, 8, 44                         # the last launch is shorter (44 = 5 x 8 + 4)
    kw = dict(device=DEV, noise="philox", seed=0, auto_reset=True, reward_mode="shaped")
    old = L.set_actor_path("tf32")
    try:
        env = VecMREnv(P * N, **kw)
        env.max_timesteps = 8
        pop = DDPGPopulation(P, seeds=SEEDS[:P], device=DEV, **_hyper_of(P))
        log = train_population(env, pop, OUNoise(P * N, device=DEV), buffer_size=2048, min_batch=64, steps=steps,
                               collect_steps=K)
        solo = []
        for p in range(P):
            e = VecMREnv(N, env_base=p * N, **kw)
            e.max_timesteps = 8
            m = _solo_learner(pop, p)
            lg = train(e, m, OUNoise(N, env_base=p * N, device=DEV), min_batch=64, steps=steps,
                       replay=ReplayBuffer(2048, 0, device=DEV), collect_steps=K)
            solo.append((lg, m))
        torch.cuda.synchronize()
    finally:
        L.set_actor_path(old)
    assert log.shape == (P, 6, 3)
    for p, (lg, m) in enumerate(solo):
        for a, b in zip(_learner_tensors(pop.member(p)), _learner_tensors(m)):
            assert torch.equal(a, b), p
        assert m.updates == pop.updates == steps
        assert np.array_equal(log[p, :, 1:], lg[:, 1:]), p
        assert np.abs(log[p, :, 0] - lg[:, 0]).max() <= 1e-12 * np.abs(lg[:, 0]).max(), p
    assert not np.array_equal(log[0], log[1])


@pytest.mark.gpu
def test_population_launches_write_nothing_outside_their_members():
    """Sentinel rows before and after every stacked array: the update writes only its members' parameter, moment and
    gradient slices (and reads the rings), the collector only the ring slots [head, head + K N) of each member, the
    members' statistics rows and its own env and OU rows."""
    from mr_rl_b200 import _lib as L
    from mr_rl_b200.ddpg import collect_population
    P, N, K = 3, 128, 3
    cap = K * N + 100
    head = 57
    s = PopSetup(P, N, torch.float64, capacity=cap, head=head)
    pop = s.pop

    def padded(t):                                         # [P, ...] -> [P + 2, ...] with sentinel rows 0 and P + 1
        buf = torch.full((P + 2, *t.shape[1:]), SENTINEL, dtype=t.dtype, device=DEV)
        buf[1:P + 1] = t
        return buf

    # ---- update, through padded copies of the state and the rings
    _fill_ring(s.rep, cap, 2)
    st = [padded(t) for t in (pop.actor, pop.actor_target, pop.critic, pop.critic_target, *pop._moments, *pop._grads)]
    pop._c.st = L.DDPGState(*[t[1].data_ptr() for t in st])
    ring = [padded(t) for t in (s.rep.s, s.rep.a, s.rep.r, s.rep.d, s.rep.s2)]
    before = [t.clone() for t in ring]
    fake = types.SimpleNamespace(members=P, random_seeds=s.rep.random_seeds, count=cap,
                                 _c=L.Replay(*[t[1].data_ptr() for t in ring], cap))
    info = torch.full((P + 2, 2), SENTINEL, dtype=torch.float32, device=DEV)
    pop._info = info[1:P + 1]
    pop.update(fake, 64)
    torch.cuda.synchronize()
    for t in st:
        assert bool((t[0] == SENTINEL).all()) and bool((t[P + 1] == SENTINEL).all())
        assert not bool((t[1:P + 1] == SENTINEL).any())
    for t, b in zip(ring, before):
        assert torch.equal(t, b)
    assert bool((info[0] == SENTINEL).all()) and bool((info[P + 1] == SENTINEL).all()) and not bool((info[1:P + 1] == SENTINEL).any())

    # ---- collector, into padded rings, statistics and OU rows
    ring = [torch.full((P + 2, *t.shape[1:]), SENTINEL, dtype=torch.float32, device=DEV) for t in (s.rep.s, s.rep.a, s.rep.r, s.rep.d, s.rep.s2)]
    fake = types.SimpleNamespace(members=P, buffer_size=cap, head=head, count=head,
                                 _c=L.Replay(*[t[1].data_ptr() for t in ring], cap))
    stats = torch.full((P + 2, 8), SENTINEL, dtype=torch.float64, device=DEV)
    stats[1:P + 1] = 0
    pop.stats = stats[1:P + 1]
    extra = 13
    x = torch.full((P * N + extra, 2), SENTINEL, dtype=torch.float64, device=DEV)
    x[:P * N] = s.noise.x_prev
    s.noise.x_prev = x
    e = s.env
    for t in (e._state, e._obs, e._sp):
        t[:, P * N:] = SENTINEL
    for t in (e._counter, e._cursor, e._status, e._done):
        t[P * N:] = 77
    collect_population(e, pop, s.noise, fake, K)
    torch.cuda.synchronize()
    owned = torch.zeros(cap, dtype=torch.bool, device=DEV)
    owned[(head + torch.arange(K * N, device=DEV)) % cap] = True
    for t in ring:
        assert bool((t[0] == SENTINEL).all()) and bool((t[P + 1] == SENTINEL).all())
        for p in range(1, P + 1):
            assert bool((t[p][~owned] == SENTINEL).all())
            assert not bool((t[p][owned] == SENTINEL).all())
    assert bool((stats[0] == SENTINEL).all()) and bool((stats[P + 1] == SENTINEL).all())
    assert bool((stats[1:P + 1, 6] == K * N).all())
    assert bool((x[P * N:] == SENTINEL).all()) and bool((x[:P * N] != SENTINEL).all())
    for t in (e._state, e._obs, e._sp):
        assert bool((t[:, P * N:] == SENTINEL).all())
    for t in (e._counter, e._cursor, e._status, e._done):
        assert bool((t[P * N:] == 77).all())
