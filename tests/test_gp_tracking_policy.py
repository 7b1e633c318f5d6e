"""GP-corrected heading control inside the fused rollout (LearningModule.tracking_policy, mr_env_rollout_gp_heading).

Without a GPU: the C struct layout, every argument error of the entry point, mr_env_rollout's rejection of the new action
source and the Python-level ValueErrors.  On the GPU: the fused policy against the step-by-step composition
vd -> predict_batch -> step (bit for bit, fp64 storage), against main.py's two-launch open-loop path, across auto-reset
boundaries, in fp32 storage, a closed loop that reaches its target, a non-finite env, and the padding behind every row."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "mr_rl_b200.h")
FAKE = C.c_void_p(256)          # a non-null address that no argument check dereferences


def test_gp_heading_policy_struct_matches_c_layout(tmp_path):
    from mr_rl_b200 import _lib as L
    prog = tmp_path / "pol.c"
    fields = [f[0] for f in L.GpHeadingPolicy._fields_]
    body = "\n".join(f'printf("{f} %zu\\n", offsetof(mr_gp_heading_policy, {f}));' for f in fields)
    prog.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "{HEADER}"\nint main(void){{{body}\n'
                    'printf("size %zu\\n", sizeof(mr_gp_heading_policy));\n'
                    'printf("src %d\\n", (int)MR_ACTIONS_GP_HEADING);return 0;}\n')
    exe = tmp_path / "pol"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert C.sizeof(L.GpHeadingPolicy) == int(out["size"])
    for f in fields:
        assert getattr(L.GpHeadingPolicy, f).offset == int(out[f]), f
    assert int(out["src"]) == L.ACTIONS_GP_HEADING == 4


def _args(n=4):
    """Arguments that pass every check of mr_env_rollout_gp_heading; the pointers are never dereferenced by the checks."""
    from mr_rl_b200 import _lib as L
    st = L.EnvState(*([FAKE] * 8), None, None, None)
    p = L.default_params()
    nz = L.Noise(L.NOISE_PHILOX, 0, None, 0, 1, 0, 0, None)
    tt = L.TimeTable(FAKE, 16, 0)
    io = L.RolloutIO()
    io.action_source, io.k_steps = L.ACTIONS_GP_HEADING, 3
    pol = L.GpHeadingPolicy(FAKE, FAKE, 8, 0, 1.4, 4.0, 0.2, -0.1, FAKE, 2.0)
    return st, p, nz, tt, io, pol


def _call(st, p, nz, tt, io, pol, n=4, dtype=0):
    from mr_rl_b200 import _lib as L
    lib = L.load()
    rc = lib.mr_env_rollout_gp_heading(C.byref(st) if st is not None else None, n, dtype, C.byref(p), C.byref(nz),
                                       C.byref(tt), C.byref(io) if io is not None else None,
                                       C.byref(pol) if pol is not None else None, None, None)
    return rc, lib.mr_last_error().decode()


def test_gp_heading_entry_point_argument_errors_need_no_gpu():
    from mr_rl_b200 import _lib as L
    st, p, nz, tt, io, pol = _args()
    rc, msg = _call(None, p, nz, tt, io, pol)
    assert rc == -1 and "mr_env_rollout_gp_heading: null state" in msg
    rc, msg = _call(st, p, nz, tt, None, pol)
    assert rc == -1 and "bad io" in msg
    rc, msg = _call(st, p, nz, tt, io, None)
    assert rc == -1 and "null policy" in msg
    for field in ("coef_x", "coef_y"):
        bad = L.GpHeadingPolicy.from_buffer_copy(pol)
        setattr(bad, field, None)
        rc, msg = _call(st, p, nz, tt, io, bad)
        assert rc == -1 and "null coefficients" in msg
    bad = L.GpHeadingPolicy.from_buffer_copy(pol)
    bad.ref = None
    rc, msg = _call(st, p, nz, tt, io, bad)
    assert rc == -1 and "null ref" in msg
    for nc in (0, -1, 4097):
        bad = L.GpHeadingPolicy.from_buffer_copy(pol)
        bad.n_coef = nc
        rc, msg = _call(st, p, nz, tt, io, bad)
        assert rc == -1 and "n_coef" in msg
    for field in ("a0", "freq", "drift_x", "drift_y", "gain"):
        for v in (math.nan, math.inf):
            bad = L.GpHeadingPolicy.from_buffer_copy(pol)
            setattr(bad, field, v)
            rc, msg = _call(st, p, nz, tt, io, bad)
            assert rc == -1 and "must be finite" in msg, field
    for src in (L.ACTIONS_TENSOR, L.ACTIONS_PHILOX, L.ACTIONS_ACTOR, L.ACTIONS_BROADCAST):
        io2 = L.RolloutIO.from_buffer_copy(io)
        io2.action_source = src
        rc, msg = _call(st, p, nz, tt, io2, pol)
        assert rc == -1 and "MR_ACTIONS_GP_HEADING" in msg
    st2 = L.EnvState.from_buffer_copy(st)
    st2.a0 = st2.noise_var = st2.is_mismatched = FAKE.value
    rc, msg = _call(st2, p, nz, tt, io, pol)
    assert rc == -3 and "per-env parameter rows" in msg
    rc, msg = _call(st, p, nz, L.TimeTable(None, 0, 0), io, pol)
    assert rc == -1 and "time table" in msg


def test_plain_rollout_still_rejects_the_gp_heading_source():
    from mr_rl_b200 import _lib as L
    st, p, nz, tt, io, _ = _args()
    lib = L.load()
    rc = lib.mr_env_rollout(C.byref(st), 4, 0, C.byref(p), C.byref(nz), C.byref(tt), C.byref(io), None, None)
    assert rc == -1 and b"mr_env_rollout: unknown action source 4" in lib.mr_last_error()


def test_tracking_policy_value_errors_need_no_gpu():
    from mr_rl_b200 import LearningModule
    lm = LearningModule.__new__(LearningModule)          # no fit, no device: only the checks run
    lm.device, lm.a0, lm.freq, lm.Dx, lm.Dy = "cpu", 1.4, 4.0, 0.0, 0.0
    lm._cheb = None
    with pytest.raises(ValueError, match="predict_batch"):
        lm.tracking_policy(np.zeros((5, 4)))
    lm._cheb = torch.zeros(2, 3, dtype=torch.float64)
    for bad in (np.zeros((5, 3)), np.zeros(4), np.zeros((0, 4)), np.zeros((2, 5, 4))):
        with pytest.raises(ValueError, match=r"\[K, 4\]"):
            lm.tracking_policy(bad)
    r = np.zeros((5, 4))
    r[2, 1] = np.nan
    with pytest.raises(ValueError, match="finite"):
        lm.tracking_policy(r)
    pol = lm.tracking_policy(np.ones((5, 4)), gain=2.0)
    assert pol.k_steps == 5 and pol.gain == 2.0 and pol.ref.dtype == torch.float64 and pol.ref.is_contiguous()


# ---------------------------------------------------------------------------------------------------------------------
# GPU

DEV = "cuda:0"
A0_SIM, SIGMA = 1.5, 0.5


@pytest.fixture(scope="module")
def lm(golden_gp):
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, WhiteKernel
    from mr_rl_b200 import LearningModule
    g = golden_gp
    X = g["X"].reshape(-1, 1)
    gX = GaussianProcessRegressor(kernel=RBF(0.2) + WhiteKernel(0.008), optimizer=None).fit(X, g["yx"])
    gY = GaussianProcessRegressor(kernel=RBF(0.25) + WhiteKernel(0.008), optimizer=None).fit(X, g["yy"])
    a0, freq, Dx, Dy = g["hyper"]
    m = LearningModule(device=DEV)
    m.set_models(gX, gY, a0, freq, Dx, Dy)
    assert m._cheb is not None
    return m


def desired_ref(lm, K):
    """A desired path as main.py builds one: fixed speed a0 freq, a turning heading, positions accumulated over dt."""
    dt = 0.030
    th = np.linspace(0.3, -2.0, K)
    v = lm.a0 * lm.freq * np.stack([np.cos(th), np.sin(th)], 1)
    p = np.vstack([np.zeros(2), np.cumsum(v * dt, 0)[:-1]])
    return np.hstack([p, v])


def make_env(n, dtype=torch.float64, noise="philox", z=None, **kw):
    from mr_rl_b200 import VecMREnv
    return VecMREnv(n, device=DEV, dtype=dtype, noise=noise, seed=7, **({"noise_table": z} if noise == "table" else {}), **kw)


def starts(n, seed=0, spread=3.0):
    rng = np.random.default_rng(seed)
    return rng.uniform(-spread, spread, (n, 2)).astype(np.float32).astype(np.float64)


def fused(lm, env, ref, gain, k_steps=None):
    res = env.rollout(policy=lm.tracking_policy(ref, gain), k_steps=k_steps, record_episodes=True)
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy().copy() if torch.is_tensor(v) else v) for k, v in res.items()}


def composed(lm, env, ref, gain, K):
    """The controller built by hand, one control step at a time: vd from env.last_pos, predict_batch, env.step."""
    r = torch.as_tensor(ref, device=DEV, dtype=torch.float64)
    acts, xy, done = [], [], []
    for k in range(K):
        pos = env.last_pos.to(torch.float64)
        vd = r[k, 2:] + gain * (r[k, :2] - pos)
        alpha = lm.predict_batch(vd)[0]
        a = torch.stack([torch.full_like(alpha, float(lm.freq)), alpha], 1)
        _, _, d, _ = env.step(a)
        acts.append(a.cpu().numpy())
        xy.append(env.last_pos.to(torch.float64).cpu().numpy().T.copy())
        done.append(d.cpu().numpy().copy())
    return np.stack(acts), np.stack(xy), np.stack(done)


def state_of(env):
    return {"state": env._state[:, :env.num_envs].cpu().numpy(), "counter": env.counter.cpu().numpy(),
            "cursor": env._cursor[:env.num_envs].cpu().numpy(), "status": env.status.cpu().numpy()}


def assert_same_state(a, b):
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.gpu
@pytest.mark.parametrize("noise,gain,n", [("philox", 0.0, 1000), ("philox", 3.0, 1000), ("table", 3.0, 1000),
                                         ("philox", 3.0, 48000)])    # 375 CTAs: the register-capped kernel
def test_fused_policy_equals_composed_controller_bit_for_bit(lm, noise, gain, n):
    K = 40
    ref = desired_ref(lm, K)
    z = np.random.default_rng(3).standard_normal((400 * K, n)) if noise == "table" else None
    init = starts(n)
    envs = []
    for _ in range(2):
        e = make_env(n, noise=noise, z=z)
        e.reset(init=init, noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
        envs.append(e)
    f = fused(lm, envs[0], ref, gain)
    acts, xy, done = composed(lm, envs[1], ref, gain, K)
    assert np.array_equal(f["actions_traj"], acts)
    assert np.array_equal(f["xy"], xy)
    assert np.array_equal(f["done_traj"], done)
    assert_same_state(state_of(envs[0]), state_of(envs[1]))
    if noise == "philox":
        assert int(envs[0].status.max()) == 0
    assert np.all(acts[:, :, 0] == lm.freq)


@pytest.mark.gpu
def test_open_loop_equals_predict_batch_then_broadcast_rollout(lm):
    n, K = 777, 48
    ref = desired_ref(lm, K)
    init = starts(n, 1)
    e1, e2 = make_env(n), make_env(n)
    for e in (e1, e2):
        e.reset(init=init, noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
    f = fused(lm, e1, ref, 0.0)
    alpha = lm.predict_batch(ref[:, 2:])[0]                                   # main.py: all K corrected headings at once
    acts = torch.stack([torch.full_like(alpha, float(lm.freq)), alpha], 1)
    r2 = e2.rollout(actions=acts, record=True)
    assert np.array_equal(f["xy"], r2["xy"].cpu().numpy())
    assert np.array_equal(f["actions_traj"], np.broadcast_to(acts.cpu().numpy()[:, None, :], (K, n, 2)))
    assert_same_state(state_of(e1), state_of(e2))


@pytest.mark.gpu
def test_policy_across_episode_boundaries(lm):
    n, K, gain = 600, 40, 2.0
    ref = desired_ref(lm, K)
    init = starts(n, 2)
    e1, e2 = make_env(n, auto_reset=True), make_env(n, auto_reset=True)
    for e in (e1, e2):
        e.max_timesteps = 12
        e.reset(init=init, noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
    f = fused(lm, e1, ref, gain)
    acts, xy, done = composed(lm, e2, ref, gain, K)
    assert (f["done_traj"].sum(0) >= 2).all()                                # at least two boundaries in every env
    assert np.array_equal(f["done_traj"], done)
    assert np.array_equal(f["actions_traj"], acts)
    live = np.broadcast_to((done == 0)[:, None, :], xy.shape)
    assert np.array_equal(f["xy"][live], xy[live])                            # composed last_pos is post-reset at a boundary
    assert_same_state(state_of(e1), state_of(e2))
    # after a reset the next heading comes from the new episode's start position
    k, i = np.argwhere(f["done_traj"][:-1] != 0)[0]
    r = torch.as_tensor(ref, device=DEV)
    p0 = torch.as_tensor(f["reset_xy"][k, :, i], device=DEV)
    alpha = lm.predict_batch((r[k + 1, 2:] + gain * (r[k + 1, :2] - p0)).reshape(1, 2))[0]
    assert float(alpha[0]) == f["actions_traj"][k + 1, i, 1]


@pytest.mark.gpu
def test_fp32_storage_agrees_with_fp64(lm):
    n, K, gain = 1000, 40, 3.0
    ref = desired_ref(lm, K)
    init = starts(n, 4)
    out = {}
    for dt in (torch.float64, torch.float32):
        e = make_env(n, dtype=dt)
        e.reset(init=init, noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
        out[dt] = fused(lm, e, ref, gain)
    a, b = out[torch.float32]["xy"].astype(np.float64), out[torch.float64]["xy"]
    assert np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0)) < 1e-4
    assert np.array_equal(out[torch.float32]["done_traj"], out[torch.float64]["done_traj"])


@pytest.mark.gpu
def test_closed_loop_reaches_the_target():
    """Noise-free matched simulator, a GP of small residuals, v_ref = 0 and a fixed target: every env ends within two step
    lengths (a0 freq dt each) of the target — fixed speed with heading-only control circles the point instead of stopping."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, WhiteKernel
    from mr_rl_b200 import LearningModule
    X = np.linspace(-np.pi, np.pi, 120).reshape(-1, 1)
    gX = GaussianProcessRegressor(kernel=RBF(0.6) + WhiteKernel(1e-4), optimizer=None).fit(X, 0.02 * np.sin(X[:, 0]))
    gY = GaussianProcessRegressor(kernel=RBF(0.6) + WhiteKernel(1e-4), optimizer=None).fit(X, -0.015 * np.cos(2 * X[:, 0]))
    m = LearningModule(device=DEV)
    m.set_models(gX, gY, 1.4, 4.0, 0.0, 0.0)
    assert m._cheb is not None
    n, dt, target = 512, 0.030, np.array([200.0, 150.0])
    step_len = m.a0 * m.freq * dt
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False)
    dist = np.linspace(0.5, 8.0, n)
    init = target + dist[:, None] * np.stack([np.cos(ang), np.sin(ang)], 1)
    K = int(np.ceil(dist.max() / step_len)) + 40
    ref = np.zeros((K, 4))
    ref[:, :2] = target
    e = make_env(n, noise="none")
    e.reset(init=init, noise_var=0.0, a0=m.a0, is_mismatched=False)
    e.rollout(policy=m.tracking_policy(ref, gain=5.0), accumulate_stats=False)
    d = np.hypot(*(e.last_pos.cpu().numpy() - target).T)
    assert d.max() <= 2 * step_len, d.max()
    e.check_status()


@pytest.mark.gpu
def test_non_finite_env_is_flagged_and_leaves_the_others_untouched(lm):
    n, K, gain, bad = 300, 16, 3.0, 37
    ref = desired_ref(lm, K)
    init = starts(n, 5)
    init_nan = init.copy()
    init_nan[bad] = np.nan
    e_ok, e_fused, e_comp = make_env(n), make_env(n), make_env(n)
    e_ok.reset(init=init, noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
    for e in (e_fused, e_comp):
        e.reset(init=init_nan, noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
    f_ok = fused(lm, e_ok, ref, gain)
    f = fused(lm, e_fused, ref, gain)
    acts, _, _ = composed(lm, e_comp, ref, gain, K)
    st_f, st_c, st_ok = state_of(e_fused), state_of(e_comp), state_of(e_ok)
    assert st_f["status"][bad] != 0 and st_f["status"][bad] == st_c["status"][bad]
    assert np.array_equal(f["actions_traj"][:, bad], acts[:, bad], equal_nan=True)   # what the standalone search returns
    keep = np.arange(n) != bad
    for k in st_ok:
        assert np.array_equal(st_f[k][..., keep], st_ok[k][..., keep]), k
    assert np.array_equal(f["xy"][..., keep], f_ok["xy"][..., keep])


@pytest.mark.gpu
def test_policy_rollout_writes_nothing_outside_its_rows(lm):
    """Sentinels behind the state rows and behind every trajectory row stay untouched (both storage types)."""
    from mr_rl_b200 import _lib as L
    n, K, pad = 128 * 5 + 37, 6, 64
    ref = torch.as_tensor(desired_ref(lm, K), device=DEV)
    pol, keep = lm.tracking_policy(ref, 2.0).c_policy(torch.device(DEV))
    for dt in (torch.float64, torch.float32):
        e = make_env(n, dtype=dt, auto_reset=True)
        e.max_timesteps = 3
        rows = {"state": e._state, "obs": e._obs, "sp": e._sp, "rew": e._rew, "done": e._done, "counter": e._counter,
                "cursor": e._cursor, "status": e._status}
        for t in rows.values():
            t[..., n:] = 77
        e.reset(init=starts(n, 6), noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
        traj = {"traj_xy": (K * 2 * n, dt), "traj_state_prime": (K * 2 * n, dt), "traj_done": (K * n, torch.uint8),
                "traj_actions": (K * n * 2, dt), "traj_rew": (K * n, dt), "traj_reset_xy": (K * 2 * n, dt),
                "traj_episode": (K * n, torch.int32), "traj_step": (K * n, torch.int32), "episode_counter": (n, torch.int32)}
        bufs = {}
        io = L.RolloutIO()
        io.action_source, io.k_steps = L.ACTIONS_GP_HEADING, K
        for name, (m, t) in traj.items():
            b = torch.full((m + pad,), 77, dtype=t, device=DEV)
            if name == "episode_counter":
                b[:n] = 0
            bufs[name] = b
            setattr(io, name, b.data_ptr())
        stats = torch.zeros(L.STATS_LEN, dtype=torch.float64, device=DEV)
        io.stats = stats.data_ptr()
        nz = e._noise_for(e.params.noise_var)
        rc = e.lib.mr_env_rollout_gp_heading(C.byref(e._c_state), n, e._dt, C.byref(e.params), C.byref(nz), C.byref(e._c_tt),
                                             C.byref(io), C.byref(pol), C.byref(e._c_out), None)
        L.check(rc, "mr_env_rollout_gp_heading")
        torch.cuda.synchronize()
        for name, (m, _) in traj.items():
            assert bool((bufs[name][m:] == 77).all()), (name, dt)
        for name, t in rows.items():
            assert bool((t[..., n:] == 77).all()), (name, dt)
        assert float(stats[L.STAT_NAMES.index("episodes")]) > 0


@pytest.mark.gpu
def test_rollout_policy_python_errors(lm):
    from mr_rl_b200 import MRLibraryError
    pol = lm.tracking_policy(desired_ref(lm, 10), 1.0)
    e = make_env(64)
    e.reset(init=starts(64), noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
    with pytest.raises(ValueError, match="k_steps"):
        e.rollout(policy=pol, k_steps=11)
    r = e.rollout(policy=pol, k_steps=4, record=True)
    assert r["xy"].shape == (4, 2, 64) and int(e.counter[0]) == 4
    e2 = make_env(64, per_env_params=True)
    e2.reset(init=starts(64), noise_var=SIGMA, a0=A0_SIM, is_mismatched=True)
    with pytest.raises(MRLibraryError, match="per-env parameter rows"):
        e2.rollout(policy=pol)
