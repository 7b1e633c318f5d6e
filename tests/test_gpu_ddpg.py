"""DDPG learner on the device (csrc/mr_ddpg.cu, mr_rl_b200/ddpg.py) against the torch restatement of the reference's
TensorFlow graph (oracle/ddpg_oracle.py — parity unpinned: no TensorFlow here).  fp32 on both sides; the tolerances
below are fp32 summation-order noise after a few Adam steps."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

BOUND = (20.0, 2 * math.pi)


def make_pair(seed=0, ref_dtype=torch.float32, **kw):
    from mr_rl_b200.actor import init_actor
    from mr_rl_b200.ddpg import DDPGLearner, init_critic
    from oracle.ddpg_oracle import DDPGOracle
    a, c, at, ct = init_actor(seed), init_critic(seed + 1), init_actor(seed + 2), init_critic(seed + 3)
    dev = DDPGLearner(a, c, BOUND, actor_target_init=at, critic_target_init=ct, device="cuda:0", **kw)
    ref = DDPGOracle(a, c, at, ct, BOUND, dtype=ref_dtype, **kw)
    return dev, ref





def fill_replay(n, seed=0):
    from mr_rl_b200.ddpg import ReplayBuffer
    g = torch.Generator().manual_seed(seed)
    rb = ReplayBuffer(n, 0, device="cuda:0")
    xy = (torch.rand(n, 2, generator=g) * 2 - 1) * 80
    s = torch.cat([xy, torch.zeros(n, 2), xy.norm(dim=1, keepdim=True)], 1)
    a = torch.rand(n, 2, generator=g) * torch.tensor(BOUND)
    xy2 = xy + torch.randn(n, 2, generator=g)
    s2 = torch.cat([xy2, torch.zeros(n, 2), xy2.norm(dim=1, keepdim=True)], 1)
    r = torch.where(torch.rand(n, generator=g) < 0.2, torch.tensor(-50.0), torch.tensor(10.0))
    d = (torch.rand(n, generator=g) < 0.15).float()
    for dst, src in ((rb.s, s), (rb.a, a), (rb.r, r), (rb.d, d), (rb.s2, s2)):
        dst.copy_(src)
    rb.count = n
    return rb, (s, a, r, d, s2)


def assert_params_close(dev, ref, atol=3e-6, rtol=2e-4):
    for name, got, want in (("actor", dev.actor_params(), ref.actor), ("actor_t", dev.actor_params(True), ref.actor_t),
                            ("critic", dev.critic_params(), ref.critic), ("critic_t", dev.critic_params(True), ref.critic_t)):
        for k, w in want.items():
            g = got[k]
            assert torch.allclose(g, w.reshape(g.shape).float(), atol=atol, rtol=rtol), \
                f"{name}.{k}: max abs diff {float((g - w.reshape(g.shape)).abs().max()):.3e}"


@pytest.mark.parametrize("batch", [64, 50, 256, 1000, 4096])
def test_update_matches_torch_restatement(batch):
    """batch <= 64: the one-launch single-CTA kernel; above: the data-parallel path (one CTA per SM, partial gradients
    summed in a fixed order) — same numbers either way."""
    dev, ref = make_pair(0)
    rb, (s, a, r, d, s2) = fill_replay(max(1000, batch), seed=batch)
    g = torch.Generator().manual_seed(5)
    for it in range(6):
        idx = torch.randperm(max(1000, batch), generator=g)[:batch]
        info = dev.update(rb, indices=idx.cuda()).cpu()
        loss, qm = ref.update(s[idx], a[idx], r[idx], d[idx], s2[idx])
        assert abs(float(info[0]) - loss) <= 1e-4 * abs(loss) + 1e-5, (it, float(info[0]), loss)
        assert abs(float(info[1]) - qm) <= 1e-4 * abs(qm) + 1e-5
    if batch <= 1000:
        assert_params_close(dev, ref)
    else:
        # Thousands of samples per update make "ReLU knife-edge" events likely: a pre-activation within fp32 rounding
        # of zero flips the mask of one hidden unit in one implementation, and Adam's normalisation turns that into a
        # visible step for that unit's ~40 parameters.  Measured over seeds (tools history): it happens to torch's own
        # fp32 run against float64 as often as to the device.  So judge against the same update in float64, robustly:
        # nearly all parameters agree to fp32 noise, at most one or two units may have taken a different branch.
        _, ref64 = make_pair(0, ref_dtype=torch.float64)
        g = torch.Generator().manual_seed(5)
        for it in range(6):
            idx = torch.randperm(max(1000, batch), generator=g)[:batch]
            ref64.update(s[idx], a[idx], r[idx], d[idx], s2[idx])
        for got, r64 in ((dev.actor_params(), ref64.actor), (dev.critic_params(), ref64.critic),
                         (dev.actor_params(True), ref64.actor_t), (dev.critic_params(True), ref64.critic_t)):
            err = torch.cat([(got[k].double() - r64[k].reshape(got[k].shape)).abs().reshape(-1) for k in r64])
            assert float(err.median()) < 5e-7 and float((err > 1e-5).double().mean()) < 0.03 and float(err.max()) < 5e-3
    # the unused t1 bias never moves, the moving statistics stay frozen
    assert torch.all(dev.critic_params()["t1b"] == 0) and torch.all(dev.critic_params()["vc"] == 1)
    assert torch.all(dev.actor_params()["m1"] == 0) and torch.all(dev.actor_params()["v2"] == 1)


def test_targets_start_from_the_soft_update_of_independent_inits():
    dev, ref = make_pair(3)
    assert_params_close(dev, ref, atol=1e-7, rtol=1e-6)
    assert not torch.allclose(dev.actor_params()["w2"], dev.actor_params(True)["w2"])


def test_internal_sampling_without_replacement_and_determinism():
    from mr_rl_b200.ddpg import DDPGLearner
    # count == batch: a sample without replacement is the whole buffer -> equals the explicit full batch
    rb, _ = fill_replay(128, seed=1)
    a, _ = make_pair(1)
    b, _ = make_pair(1)
    ia = a.update(rb, 128).clone()
    ib = b.update(rb, indices=torch.arange(128)).clone()
    assert torch.allclose(ia, ib, rtol=1e-5, atol=1e-6)
    for k, v in a.critic_params().items():
        assert torch.allclose(v, b.critic_params()[k], atol=2e-6, rtol=1e-4), k
    # same seed and update index -> same minibatch; the next update draws another one
    rb, _ = fill_replay(5000, seed=2)
    c, _ = make_pair(2)
    e, _ = make_pair(2)
    i1, i2 = c.update(rb, 64).clone(), e.update(rb, 64).clone()
    assert torch.equal(i1, i2) and torch.equal(c.critic, e.critic)
    i3 = c.update(rb, 64).clone()
    assert not torch.equal(i1, i3)


def test_update_argument_errors():
    from mr_rl_b200 import _lib as L
    dev, _ = make_pair(0)
    rb, _ = fill_replay(100)
    rb.count = 10
    with pytest.raises(L.MRLibraryError, match="min_batch|count"):
        dev.update(rb, 64)
    assert dev.updates == 0
    rb.count = 100
    with pytest.raises(L.MRLibraryError, match="batch"):
        dev.update(rb, 0)


def test_replay_ring_add_wraps_like_the_deque():
    from mr_rl_b200.ddpg import ReplayBuffer
    rb = ReplayBuffer(8, device="cuda:0")
    stride = 256
    for step in range(3):                                   # 3 x 3 transitions into 8 slots: the oldest one is dropped
        obs = torch.zeros(5, stride, dtype=torch.float64, device="cuda:0")
        obs2 = torch.zeros(5, stride, dtype=torch.float64, device="cuda:0")
        for k in range(5):
            obs[k, :3] = torch.arange(3, device="cuda:0") + 10 * step + 100 * k
            obs2[k, :3] = obs[k, :3] + 0.5
        act = (torch.arange(6, dtype=torch.float64, device="cuda:0").reshape(3, 2) + step)
        rew = torch.full((3,), float(step), dtype=torch.float64, device="cuda:0")
        done = torch.tensor([0, 1, 0], dtype=torch.uint8, device="cuda:0")
        rb.add(obs, act, rew, done, obs2, 3)
    assert rb.size() == 8 and rb.head == 1
    s = rb.s.cpu()
    # slot 0 was overwritten by the last transition of step 2; slots 1, 2 still hold step 0's transitions 1, 2
    assert s[0].tolist() == [22.0, 122.0, 222.0, 322.0, 422.0]
    assert s[1].tolist() == [1.0, 101.0, 201.0, 301.0, 401.0]
    assert s[6].tolist() == [20.0, 120.0, 220.0, 320.0, 420.0]
    assert rb.s2.cpu()[7, 0] == 21.5 and rb.r.cpu()[7] == 2.0 and rb.d.cpu().tolist()[6:8] == [0.0, 1.0]
    assert rb.a.cpu()[0].tolist() == [6.0, 7.0]


def test_ou_noise_follows_the_reference_recurrence():
    from mr_rl_b200.ddpg import OUNoise
    n = 200_000
    ou = OUNoise(n, sigma=0.3, theta=0.15, dt=1e-2, seed=4, device="cuda:0")
    act = torch.zeros(n, 2, dtype=torch.float64, device="cuda:0")
    ou.add_to(act)
    x1 = ou.x_prev.clone()
    assert torch.equal(act, x1)                                              # x0 = 0: the first sample is sigma sqrt(dt) z
    z = x1 / (0.3 * math.sqrt(1e-2))
    assert abs(float(z.mean())) < 0.01 and abs(float(z.std()) - 1) < 0.01
    assert abs(float((z[:, 0] * z[:, 1]).mean())) < 0.01
    base = torch.ones(n, 2, dtype=torch.float32, device="cuda:0")
    ou.add_to(base)
    incr = (ou.x_prev - (x1 + 0.15 * (0.0 - x1) * 1e-2)) / (0.3 * math.sqrt(1e-2))   # the second normal draw
    assert abs(float(incr.std()) - 1) < 0.01 and abs(float((incr * z).mean())) < 0.01
    assert torch.allclose(base.double(), 1 + ou.x_prev, atol=1e-6)
    ou2 = OUNoise(n, seed=4, device="cuda:0")
    act2 = torch.zeros(n, 2, dtype=torch.float64, device="cuda:0")
    ou2.add_to(act2)
    assert torch.equal(act2, x1)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_vectorised_training_loop_runs_and_learns_something(dt):
    from mr_rl_b200 import VecMREnv
    from mr_rl_b200.ddpg import DDPGLearner, OUNoise, ReplayBuffer, train
    env = VecMREnv(256, device="cuda:0", dtype=dt, noise="philox", seed=0, auto_reset=True)
    learner = DDPGLearner(device="cuda:0", seed=0)
    before = learner.actor.clone()
    rb = ReplayBuffer(10000, 0, device="cuda:0")
    log = train(env, learner, OUNoise(256, device="cuda:0"), min_batch=64, steps=40, replay=rb)
    assert log.shape == (40, 3) and np.isfinite(log).all()
    assert rb.size() == 10000 and learner.updates == 40
    assert not torch.equal(before, learner.actor) and torch.isfinite(learner.actor).all() and torch.isfinite(learner.critic).all()
    # the critic learns the scale of the returns: its loss drops from the first updates
    assert log[-5:, 1].mean() < log[:5, 1].mean()
    env.check_status()
    # what went into the ring is what the env produced: states are [x, y, 0, 0, d] rows, rewards the constant 10
    s = rb.s.cpu().numpy()
    assert np.allclose(s[:, 4], np.hypot(s[:, 0], s[:, 1]), rtol=1e-6) and np.all(s[:, 2:4] == 0)
    assert np.all(rb.r.cpu().numpy() == 10.0) and set(np.unique(rb.d.cpu().numpy())) <= {0.0, 1.0}


def test_training_loop_reproduces_the_reference_warmup_quirk():
    """RL/MR_ddpg.py:281-284: while the buffer holds fewer than min_batch transitions the loop `continue`s before
    `state = next_state`, so the stored state `s` (and the policy input) stays the observation of the last reset while the
    env moves on.  stale_state_warmup=True reproduces it; the default advances the state every iteration."""
    from mr_rl_b200 import VecMREnv
    from mr_rl_b200.ddpg import DDPGLearner, OUNoise, ReplayBuffer, train
    n, min_batch = 2, 12
    for stale in (True, False):
        env = VecMREnv(n, device="cuda:0", noise="philox", seed=5, auto_reset=True)
        rb = ReplayBuffer(1000, 0, device="cuda:0")
        train(env, DDPGLearner(device="cuda:0", seed=0), OUNoise(n, device="cuda:0"), min_batch=min_batch, steps=8, replay=rb,
              stale_state_warmup=stale)
        s, s2 = rb.s.cpu().numpy(), rb.s2.cpu().numpy()
        reset_obs = s[:n]
        warm = min_batch // n                                  # iterations whose transitions are stored before the first update
        if stale:
            for it in range(warm):
                assert np.array_equal(s[it * n:(it + 1) * n], reset_obs), it
            assert np.array_equal(s[warm * n:(warm + 1) * n], s2[(warm - 1) * n:warm * n])   # then state = next_state
        else:
            for it in range(1, warm + 1):
                assert np.array_equal(s[it * n:(it + 1) * n], s2[(it - 1) * n:it * n]), it
            assert not np.array_equal(s[n:2 * n], reset_obs)


def test_replay_ring_keeps_what_the_reference_deque_keeps():
    """The same 11 transitions pushed through RL/MR_ddpg.py's ReplayBuffer(8) (golden ddpg_host.npz) and through the
    device ring: the same transitions survive the overflow, the size saturates at the capacity."""
    from conftest import Golden
    from mr_rl_b200.ddpg import OUNoise, ReplayBuffer
    g = Golden("ddpg_host.npz")
    rb = ReplayBuffer(8, 0, device="cuda:0")
    ids = np.arange(11, dtype=np.float64)
    for lo, hi in ((0, 4), (4, 8), (8, 11)):
        k = torch.as_tensor(ids[lo:hi], device="cuda:0")
        obs = k.repeat(5, 1).contiguous()                              # SoA rows [5][m]
        rb.add(obs, torch.stack([k, -k], 1).contiguous(), 10.0 + k, (k % 3 == 0).to(torch.uint8), (obs + 0.5).contiguous(), hi - lo)
    assert rb.size() == int(g["size"])
    stored = np.sort(rb.r.cpu().numpy().astype(np.float64) - 10.0)
    assert np.array_equal(stored, np.sort(g["kept"]))
    row = {float(r - 10.0): i for i, r in enumerate(rb.r.cpu().numpy())}
    i9 = row[9.0]
    assert rb.s.cpu()[i9].tolist() == [9.0] * 5 and rb.s2.cpu()[i9].tolist() == [9.5] * 5
    assert rb.a.cpu()[i9].tolist() == [9.0, -9.0] and rb.d.cpu()[i9] == 1.0
    # the device OU process uses the reference's default parameters
    ou = OUNoise(4, device="cuda:0")
    assert (ou.theta, ou.sigma, ou.dt) == tuple(g["ou_params"])


def test_parallel_sampler_draws_distinct_uniform_rows():
    """mr_replay_sample: a keyed bijection walked into [0, count) — every batch is duplicate-free, in range, reproducible,
    changes with the update index, and covers the ring evenly."""
    from mr_rl_b200.ddpg import ReplayBuffer
    for count, batch in ((64, 64), (1000, 64), (10000, 4096), (1 << 20, 65536), (3, 2)):
        rb = ReplayBuffer(max(count, 4), 7, device="cuda:0")
        rb.count = count
        a = rb.sample_indices(batch, 1).cpu().numpy()
        assert a.min() >= 0 and a.max() < count and len(np.unique(a)) == batch
        assert np.array_equal(a, rb.sample_indices(batch, 1).cpu().numpy())
        if count > 64:
            assert not np.array_equal(a, rb.sample_indices(batch, 2).cpu().numpy())
    rb = ReplayBuffer(10000, 3, device="cuda:0")
    rb.count = 10000
    hits = np.zeros(10000)
    for u in range(1, 401):
        hits[rb.sample_indices(250, u).cpu().numpy()] += 1               # 100000 draws over 10000 rows: mean 10 per row
    assert abs(hits.mean() - 10.0) < 1e-9 and 2.8 < hits.std() < 3.5   # binomial(400, 1/40): sigma = 3.12
    assert hits.max() < 30 and (hits == 0).sum() < 10


def test_wide_update_with_internal_sampling_is_deterministic():
    rb, _ = fill_replay(50000, seed=9)
    a, _ = make_pair(4)
    b, _ = make_pair(4)
    for _ in range(3):
        ia, ib = a.update(rb, 8192).clone(), b.update(rb, 8192).clone()
        assert torch.equal(ia, ib) and torch.isfinite(ia).all()
    assert torch.equal(a.actor, b.actor) and torch.equal(a.critic_target, b.critic_target)
    assert not torch.equal(a.actor, make_pair(4)[0].actor)


def test_split_gradient_apply_path_equals_the_fused_wide_update():
    """mr_ddpg_gradients + mr_ddpg_apply (the halves a multi-GPU learner puts its all-reduce between) on one rank ==
    mr_ddpg_update on the data-parallel path (to the last bits: the two Adam kernels may contract their FMAs differently)."""
    rb, _ = fill_replay(20000, seed=3)
    a, _ = make_pair(6)
    b, _ = make_pair(6)
    for _ in range(4):
        ia = a.update(rb, 2048).clone()
        ib = b.update_distributed(rb, 2048).clone()
        assert torch.allclose(ia, ib, rtol=1e-6, atol=1e-7)
    for x, y in ((a.actor, b.actor), (a.critic, b.critic), (a.actor_target, b.actor_target), (a.critic_target, b.critic_target)):
        assert torch.allclose(x, y, rtol=1e-6, atol=1e-8)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_learner_matches_one_rank_on_the_joint_minibatch(tmp_path):
    """Two processes (one per GPU, NCCL): each takes the gradients of its own 512 rows, all-reduces, applies the mean ==
    one rank updating on the 1024 rows together (fp32 summation order aside); both ranks end with identical parameters."""
    import os
    import subprocess
    import sys
    out = tmp_path / "dist.pt"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(root, "tests", "dist_ddpg_worker.py"), str(out)]
    subprocess.run(cmd, check=True, cwd=root, timeout=300)
    res = torch.load(out)
    assert torch.equal(res["rank0_actor"], res["rank1_actor"]) and torch.equal(res["rank0_critic"], res["rank1_critic"])
    rb, _ = fill_replay(4096, seed=11)
    single, _ = make_pair(8)
    for u in range(3):
        idx = torch.cat([res["idx"][0][u], res["idx"][1][u]])
        single.update(rb, indices=idx.cuda())
    assert torch.allclose(single.critic.cpu(), res["rank0_critic"], atol=3e-6, rtol=2e-4)
    assert torch.allclose(single.actor.cpu(), res["rank0_actor"], atol=3e-6, rtol=2e-4)
