"""DDPG experience collection inside the fused rollout (ddpg.collect, mr_env_rollout_ddpg_collect).

Without a GPU: the C struct layout, every argument error of the entry point and the Python-level ValueErrors.  On the
GPU: one collect launch against K rounds of predict -> add_to -> step -> add (bit for bit on the 3xTF32 actor path,
Philox and table noise, fp64 and fp32 storage, through auto resets), a launch that wraps the ring, the default 3xFP16
path, train(collect_steps=1) against train(), training with K > 1, and the memory a launch does not own."""
import ctypes as C
import math
import os
import subprocess
import types

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_err

HEADER = os.path.join(ROOT, "include", "mr_rl_b200.h")
FAKE = C.c_void_p(256)          # a non-null address that no argument check dereferences


def test_collect_struct_matches_c_layout(tmp_path):
    from mr_rl_b200 import _lib as L
    prog = tmp_path / "col.c"
    fields = [f[0] for f in L.DDPGCollect._fields_]
    body = "\n".join(f'printf("{f} %zu\\n", offsetof(mr_ddpg_collect, {f}));' for f in fields)
    prog.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "{HEADER}"\nint main(void){{{body}\n'
                    'printf("size %zu\\n", sizeof(mr_ddpg_collect));\n'
                    'printf("ring_size %zu\\n", sizeof(mr_replay));return 0;}\n')
    exe = tmp_path / "col"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert C.sizeof(L.DDPGCollect) == int(out["size"])
    assert C.sizeof(L.Replay) == int(out["ring_size"])
    for f in fields:
        assert getattr(L.DDPGCollect, f).offset == int(out[f]), f


def _args():
    """Arguments that pass every check of mr_env_rollout_ddpg_collect; the pointers are never dereferenced by the checks."""
    from mr_rl_b200 import _lib as L
    st = L.EnvState(*([FAKE] * 8), None, None, None)
    p = L.default_params()
    nz = L.Noise(L.NOISE_PHILOX, 0, None, 0, 1, 0, 0, None)
    tt = L.TimeTable(FAKE, 16, 0)
    io = L.RolloutIO()
    io.action_source, io.k_steps, io.actor = L.ACTIONS_ACTOR, 3, FAKE.value
    ring = L.Replay(FAKE, FAKE, FAKE, FAKE, FAKE, 64)
    c = L.DDPGCollect(FAKE, 0.15, 0.0, 0.3, 1e-2, 5, 0, 0, ring, 10)
    out = L.StepOut(FAKE, FAKE, FAKE, None, 16, 0, 0)
    return st, p, nz, tt, io, c, out


def _call(st, p, nz, tt, io, c, out, n=4, dtype=0):
    from mr_rl_b200 import _lib as L
    lib = L.load()
    rc = lib.mr_env_rollout_ddpg_collect(C.byref(st) if st is not None else None, n, dtype, C.byref(p), C.byref(nz),
                                         C.byref(tt), C.byref(io) if io is not None else None,
                                         C.byref(c) if c is not None else None, C.byref(out) if out is not None else None, None)
    return rc, lib.mr_last_error().decode()


def test_collect_entry_point_argument_errors_need_no_gpu():
    from mr_rl_b200 import _lib as L
    st, p, nz, tt, io, c, out = _args()
    fn = "mr_env_rollout_ddpg_collect"
    rc, msg = _call(None, p, nz, tt, io, c, out)
    assert rc == -1 and f"{fn}: null state" in msg
    rc, msg = _call(st, p, nz, tt, None, c, out)
    assert rc == -1 and "bad io" in msg
    for src in (L.ACTIONS_TENSOR, L.ACTIONS_PHILOX, L.ACTIONS_BROADCAST, L.ACTIONS_GP_HEADING):
        io2 = L.RolloutIO.from_buffer_copy(io)
        io2.action_source = src
        rc, msg = _call(st, p, nz, tt, io2, c, out)
        assert rc == -1 and "must be MR_ACTIONS_ACTOR" in msg, src
    io2 = L.RolloutIO.from_buffer_copy(io)
    io2.actor = None
    rc, msg = _call(st, p, nz, tt, io2, c, out)
    assert rc == -1 and "null actor" in msg
    rc, msg = _call(st, p, nz, tt, io, None, out)
    assert rc == -1 and "null collect struct" in msg
    bad = L.DDPGCollect.from_buffer_copy(c)
    bad.ou_state = None
    rc, msg = _call(st, p, nz, tt, io, bad, out)
    assert rc == -1 and "null ou_state" in msg
    for field in ("s", "a", "r", "d", "s2"):
        bad = L.DDPGCollect.from_buffer_copy(c)
        setattr(bad.ring, field, None)
        rc, msg = _call(st, p, nz, tt, io, bad, out)
        assert rc == -1 and "null replay ring array" in msg, field
    for o in (None, L.StepOut(None, FAKE, FAKE, None, 16, 0, 0)):
        rc, msg = _call(st, p, nz, tt, io, c, o)
        assert rc == -1 and "out->obs" in msg
    for cap in (0, -5):
        bad = L.DDPGCollect.from_buffer_copy(c)
        bad.ring.capacity, bad.head = cap, 0
        rc, msg = _call(st, p, nz, tt, io, bad, out)
        assert rc == -1 and "capacity must be positive" in msg, cap
    for head in (-1, 64, 1000):
        bad = L.DDPGCollect.from_buffer_copy(c)
        bad.head = head
        rc, msg = _call(st, p, nz, tt, io, bad, out)
        assert rc == -1 and "0 <= head < capacity" in msg, head
    rc, msg = _call(st, p, nz, tt, io, c, out, n=65)
    assert rc == -1 and "n > capacity" in msg
    for field in ("ou_theta", "ou_mu", "ou_sigma", "ou_dt"):
        for v in (math.nan, math.inf, -math.inf):
            bad = L.DDPGCollect.from_buffer_copy(c)
            setattr(bad, field, v)
            rc, msg = _call(st, p, nz, tt, io, bad, out)
            assert rc == -1 and "must be finite" in msg, field
    rc, msg = _call(st, p, nz, L.TimeTable(None, 0, 0), io, c, out)
    assert rc == -1 and "time table" in msg
    st2 = L.EnvState.from_buffer_copy(st)
    st2.a0 = st2.noise_var = st2.is_mismatched = FAKE.value
    rc, msg = _call(st2, p, nz, tt, io, c, out)
    assert rc == -3 and "per-env parameter rows" in msg
    old = L.set_actor_path("simt")
    try:
        rc, msg = _call(st, p, nz, tt, io, c, out)
        assert rc == -3 and "CUDA-core actor path" in msg
    finally:
        L.set_actor_path(old)
    # mr_env_rollout is unchanged: the collector is only reachable through its own entry point
    lib = L.load()
    io2 = L.RolloutIO.from_buffer_copy(io)
    io2.action_source = 5
    rc = lib.mr_env_rollout(C.byref(st), 4, 0, C.byref(p), C.byref(nz), C.byref(tt), C.byref(io2), None, None)
    assert rc == -1 and b"unknown action source 5" in lib.mr_last_error()


def test_collect_python_value_errors_need_no_gpu():
    from mr_rl_b200.ddpg import collect, train
    env = types.SimpleNamespace(num_envs=8)
    with pytest.raises(ValueError, match="stale_state_warmup"):
        train(env, None, None, collect_steps=4, stale_state_warmup=True)
    with pytest.raises(ValueError, match="collect_steps must be at least 1"):
        train(env, None, None, collect_steps=0, replay=types.SimpleNamespace(buffer_size=100))
    with pytest.raises(ValueError, match="replay buffer holds"):
        train(env, None, None, collect_steps=2, replay=types.SimpleNamespace(buffer_size=7))
    with pytest.raises(ValueError, match="k_steps must be at least 1"):
        collect(env, None, None, types.SimpleNamespace(buffer_size=100), 0)
    with pytest.raises(ValueError, match="replay buffer holds"):
        collect(env, None, None, types.SimpleNamespace(buffer_size=7), 3)


# ---------------------------------------------------------------------------------------------------------------------
# GPU

DEV = "cuda:0"
SENTINEL = 77.0


def bn_actor(seed=7):
    """An actor with non-trivial batch-norm statistics and a last layer that does not saturate the tanh."""
    from mr_rl_b200 import init_actor
    params = init_actor(seed)
    g = torch.Generator().manual_seed(seed + 1)
    params["w3"] = 0.5 * torch.randn(64, 2, generator=g)
    for k in ("m1", "m2"):
        params[k] = 0.05 * torch.randn(64, generator=g)
    for k in ("v1", "v2"):
        params[k] = 0.5 + torch.rand(64, generator=g)
    for k in ("be1", "be2", "b1", "b2"):
        params[k] = 0.02 * torch.randn(64, generator=g)
    return params


class Setup:
    """env + learner + OU noise + ring, built twice from the same seeds (one for the fused launch, one for the composed loop)."""

    def __init__(self, n, dtype, noise, capacity, head, z=None, ou_rows=None, **env_kw):
        from mr_rl_b200 import VecMREnv
        from mr_rl_b200.ddpg import DDPGLearner, OUNoise, ReplayBuffer
        self.n = n
        self.env = VecMREnv(n, device=DEV, dtype=dtype, noise=noise, seed=3, auto_reset=True,
                            **({"noise_table": z} if noise == "table" else {}), **env_kw)
        self.env.max_timesteps = 5                        # episode boundaries inside the launch
        self.env.reset(noise_var=1.0, a0=1.0)
        self.learner = DDPGLearner(actor=bn_actor(), device=DEV, seed=0)
        self.noise = OUNoise(ou_rows or n, sigma=0.3, seed=11, env_base=5, device=DEV)
        self.noise.calls = 3                              # a process that has run before
        self.noise.x_prev.copy_(0.2 * torch.randn(ou_rows or n, 2, generator=torch.Generator().manual_seed(4),
                                                  dtype=torch.float64))
        self.rb = ReplayBuffer(capacity, 0, device=DEV)
        for t in (self.rb.s, self.rb.a, self.rb.r, self.rb.d, self.rb.s2):
            t.fill_(SENTINEL)
        self.rb.head, self.rb.count = head, head

    def composed(self, k):
        """K rounds of the acting loop of ddpg.train, and the episode statistics a fused launch accumulates."""
        env, n = self.env, self.n
        state = env._obs.clone()
        stats = np.zeros(8)
        for _ in range(k):
            ctr = env.counter.clone()
            a = self.learner.predict(state, n)
            self.noise.add_to(a)
            _, rew, done, _ = env.step(a)
            self.rb.add(state, a, rew, done, env._obs, n)
            state.copy_(env._obs)
            d = done.bool().cpu().numpy()
            length = (ctr + 1).cpu().numpy()[d]
            stats[0] += d.sum(); stats[1] += length.sum(); stats[2] += float(rew.double().sum())
            stats[5] += (length > env.max_timesteps).sum(); stats[6] += n
        return stats

    def snapshot(self):
        e, rb = self.env, self.rb
        return {"s": rb.s, "a": rb.a, "r": rb.r, "d": rb.d, "s2": rb.s2, "ou": self.noise.x_prev, "state": e._state,
                "counter": e._counter, "cursor": e._cursor, "status": e._status, "obs": e._obs, "rew": e._rew,
                "done": e._done}


def table_for(n, k):
    return np.random.default_rng(5).standard_normal((40 * k + 64, n))


def assert_same(f, c):
    sf, sc = f.snapshot(), c.snapshot()
    for key in sf:
        assert torch.equal(sf[key], sc[key]), key
    assert (f.rb.head, f.rb.count, f.noise.calls) == (c.rb.head, c.rb.count, c.noise.calls)


@pytest.mark.gpu
@pytest.mark.parametrize("noise", ["philox", "table"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", [1000, 300])
def test_collect_equals_composed_loop_bit_for_bit(noise, dtype, n):
    from mr_rl_b200 import _lib as L
    from mr_rl_b200.ddpg import collect
    K1, K2 = 14, 3
    z = table_for(n, K1 + K2) if noise == "table" else None
    old = L.set_actor_path("tf32")
    try:
        f = Setup(n, dtype, noise, capacity=(K1 + K2) * n + 37, head=50, z=z)
        c = Setup(n, dtype, noise, capacity=(K1 + K2) * n + 37, head=50, z=z)
        f.env.reset_stats()
        collect(f.env, f.learner, f.noise, f.rb, K1)
        collect(f.env, f.learner, f.noise, f.rb, K2)      # continues where the first launch left the ring and the noise
        stats = c.composed(K1 + K2)
        torch.cuda.synchronize()
    finally:
        L.set_actor_path(old)
    assert_same(f, c)
    assert stats[0] >= 2 * n                               # every env crossed at least two episode boundaries
    got = f.env.stats.cpu().numpy()
    for k in (0, 1, 2, 5, 6):                              # episodes, lengths, rewards (constant 10), timeouts, env-steps
        assert got[k] == stats[k], L.STAT_NAMES[k]
    assert got[0] == got[3] + got[4] + got[5] and got[7] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_collect_that_wraps_the_ring(dtype):
    """K n > capacity with the head near the end: the ring equals the one K sequential adds leave (the transitions a later
    one of the same launch overwrites are never written)."""
    from mr_rl_b200 import _lib as L
    from mr_rl_b200.ddpg import collect
    n, K = 300, 14
    cap = 5 * n + 17                                       # K n = 4200 > 1517
    old = L.set_actor_path("tf32")
    try:
        f = Setup(n, dtype, "philox", capacity=cap, head=cap - 40)
        c = Setup(n, dtype, "philox", capacity=cap, head=cap - 40)
        collect(f.env, f.learner, f.noise, f.rb, K)
        c.composed(K)
        torch.cuda.synchronize()
    finally:
        L.set_actor_path(old)
    assert_same(f, c)
    assert f.rb.count == cap and f.rb.head == (cap - 40 + K * n) % cap


@pytest.mark.gpu
def test_collect_default_fp16_path_agrees_with_the_composed_loop():
    from mr_rl_b200.ddpg import collect
    n, K = 1000, 14
    f = Setup(n, torch.float64, "philox", capacity=K * n, head=0)
    c = Setup(n, torch.float64, "philox", capacity=K * n, head=0)
    res = collect(f.env, f.learner, f.noise, f.rb, K, record=True, record_done=True, record_episodes=True)
    c.composed(K)
    torch.cuda.synchronize()
    assert torch.equal(f.noise.x_prev, c.noise.x_prev)     # the OU process does not depend on the actor
    hi = torch.tensor([20.0, 2 * math.pi], device=DEV)
    assert float(((f.rb.a - c.rb.a).abs() / hi).max()) < 1e-4
    assert rel_err(f.env.last_pos.cpu().numpy(), c.env.last_pos.cpu().numpy()) < 2e-6
    assert torch.equal(f.env.counter, c.env.counter)
    # the recorded actions are the applied ones, the same that went into the ring (slot k n + i)
    assert torch.equal(res["actions_traj"].reshape(-1, 2).float(), f.rb.a)
    assert torch.equal(res["done_traj"].reshape(-1).float(), f.rb.d)


@pytest.mark.gpu
def test_train_with_collect_steps_1_equals_train():
    from mr_rl_b200 import VecMREnv, _lib as L
    from mr_rl_b200.ddpg import DDPGLearner, OUNoise, ReplayBuffer, train
    n, iters = 256, 20
    out = []
    old = L.set_actor_path("tf32")
    try:
        for cs in (None, 1):
            env = VecMREnv(n, device=DEV, noise="philox", seed=0, auto_reset=True, reward_mode="shaped")
            env.max_timesteps = 8
            learner = DDPGLearner(actor=bn_actor(), device=DEV, seed=0)
            log = train(env, learner, OUNoise(n, device=DEV), min_batch=64, steps=iters, replay=ReplayBuffer(4096, 0, device=DEV),
                        collect_steps=cs)
            out.append((log, learner))
    finally:
        L.set_actor_path(old)
    (log0, l0), (log1, l1) = out
    assert log0.shape == log1.shape == (iters, 3)
    for a, b in ((l0.actor, l1.actor), (l0.actor_target, l1.actor_target), (l0.critic, l1.critic),
                 (l0.critic_target, l1.critic_target), *zip(l0._moments, l1._moments)):
        assert torch.equal(a, b)
    assert l0.updates == l1.updates == iters
    assert np.array_equal(log0[:, 1:], log1[:, 1:])
    assert np.abs(log0[:, 0] - log1[:, 0]).max() <= 1e-12 * np.abs(log0[:, 0]).max()
    assert np.unique(log0[:, 0]).size > 1                  # the shaped reward moves


@pytest.mark.gpu
def test_train_with_collect_steps_16_learns_something():
    from mr_rl_b200 import VecMREnv
    from mr_rl_b200.ddpg import DDPGLearner, OUNoise, ReplayBuffer, train
    n, K, launches = 256, 16, 40
    env = VecMREnv(n, device=DEV, noise="philox", seed=0, auto_reset=True, reward_mode="shaped")
    learner = DDPGLearner(device=DEV, seed=0)
    before = learner.actor.clone()
    rb = ReplayBuffer(10000, 0, device=DEV)
    log = train(env, learner, OUNoise(n, device=DEV), min_batch=64, steps=K * launches, replay=rb, collect_steps=K)
    assert log.shape == (launches, 3) and np.isfinite(log).all()
    assert rb.size() == 10000 and learner.updates == K * launches
    assert not torch.equal(before, learner.actor) and torch.isfinite(learner.actor).all() and torch.isfinite(learner.critic).all()
    # the critic learns the scale of the returns, negative under the shaped reward (-0.1 per step, -100 per timeout); its
    # loss is no yardstick here: it stays ~0 until the first timeouts reach the ring, then jumps
    assert log[-5:, 2].mean() < min(0.0, log[:5, 2].mean())
    env.check_status()
    s, s2 = rb.s.cpu().numpy(), rb.s2.cpu().numpy()
    for x in (s, s2):
        assert np.allclose(x[:, 4], np.hypot(x[:, 0], x[:, 1]), rtol=1e-6) and np.all(x[:, 2:4] == 0)
    assert set(np.unique(rb.r.cpu().numpy())) <= {-0.1, -100.0, 100.0} | {np.float32(-0.1)}
    assert set(np.unique(rb.d.cpu().numpy())) <= {0.0, 1.0}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_collect_writes_nothing_outside_what_it_owns(dtype):
    """Ring slots outside [head, head + K n), OU rows beyond n and the padding rows of the env keep their sentinels."""
    from mr_rl_b200.ddpg import collect
    n, K, extra = 300, 6, 13
    cap = K * n + 500
    head = 321
    f = Setup(n, dtype, "philox", capacity=cap, head=head, ou_rows=n + extra)
    f.noise.x_prev[n:] = SENTINEL
    e = f.env
    pad = e._np - n
    assert pad > 0
    for t in (e._state, e._obs, e._sp):
        t[:, n:] = SENTINEL
    for t in (e._rew,):
        t[n:] = SENTINEL
    for t in (e._counter, e._cursor, e._status, e._done):
        t[n:] = 77
    collect(f.env, f.learner, f.noise, f.rb, K)
    torch.cuda.synchronize()
    owned = torch.zeros(cap, dtype=torch.bool, device=DEV)
    owned[(head + torch.arange(K * n, device=DEV)) % cap] = True
    for t in (f.rb.s, f.rb.a, f.rb.r, f.rb.d, f.rb.s2):
        assert bool((t[~owned] == SENTINEL).all())
        assert not bool((t[owned] == SENTINEL).all())
    assert bool((f.noise.x_prev[n:] == SENTINEL).all()) and bool((f.noise.x_prev[:n] != SENTINEL).all())
    for t in (e._state, e._obs, e._sp):
        assert bool((t[:, n:] == SENTINEL).all())
    assert bool((e._rew[n:] == SENTINEL).all())
    for t in (e._counter, e._cursor, e._status, e._done):
        assert bool((t[n:] == 77).all())
