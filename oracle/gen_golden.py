"""TEST INFRASTRUCTURE — regenerate tests/golden/*.npz from the LIVE reference.

Run in the build container only (needs /root/reference):

    python -m oracle.gen_golden

The reference has no golden vectors for this path (SURVEY.md §4/§8c), so the pin is
the unmodified reference code itself executed here, with numpy.random.normal patched
to pop from a recorded standard-normal stream.  Library versions are stored in every
file.  Inputs (actions, init, noise stream seeds) are stored too, so the parity tests
on the GPU box need nothing but these files.
"""
from __future__ import annotations

import os

import numpy as np

from . import live_reference as lr

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
KEEP = ("pos", "obs", "done", "counter", "state_prime", "cursor", "attempts", "carry_f", "carry_h", "t", "rew",
        "reset_obs", "reset_cursor", "reset_carry_f", "reset_carry_h", "reset_state_prime")


def versions():
    import scipy
    import sklearn
    return np.array([f"numpy {np.__version__}", f"scipy {scipy.__version__}", f"scikit-learn {sklearn.__version__}"])


def random_actions(T, seed=1):
    """SURVEY §8d C1: f~U[0,20), alpha~U[0,2pi), columns drawn f then alpha."""
    rng = np.random.default_rng(seed)
    f = rng.uniform(0, 20, size=T)
    al = rng.uniform(0, 2 * np.pi, size=T)
    return np.stack([f, al], axis=1)


def circle_actions(T, freq=4.0):
    """main.py:27-29 circle sweep."""
    a = np.zeros((T, 3))
    a[:, 0] = freq
    a[:, 1] = np.linspace(-np.pi, np.pi, T)
    return a


def single_env_cases():
    """name -> (actions, init, noise_var, a0, is_mismatched, z_seed, z_len, prior)

    ``prior`` = an episode run on the same env object before the recorded one, to expose
    the reset-ordering quirk (MR_env.py:181 before :183)."""
    T = 500
    ra = random_actions(T)
    return {
        "c1_sigma0": (ra, [110.0, 105.0], 0.0, 1.0, False, 0, 64 * T, None),
        "c1_sigma1": (ra, [110.0, 105.0], 1.0, 1.0, False, 0, 64 * T, None),
        "c1_mismatch_circle": (circle_actions(T), np.array([0, 0]), 0.5, 1.5, True, 0, 64 * T, None),
        "c1_mismatch_idle": (np.zeros((100, 3)), np.array([0, 0]), 0.5, 1.5, True, 3, 100 * 1200, None),
        "c1_default_sim_params": (ra[:60], [110.0, 105.0], 0.0, 0.0, False, 0, 256 * 60, None),
        "near_goal": (ra[:60], [25.0, 20.0], 1.0, 1.0, False, 4, 256 * 60, None),
        "out_of_bounds": (np.tile([[20.0, 0.0]], (60, 1)), [4999.5, 20.0], 1.0, 1.0, False, 5, 256 * 60, None),
        "float32_init": (ra[:120], np.array([113.37, 101.91], dtype=np.float32), 1.0, 1.0, False, 6, 256 * 120, None),
        "reset_after_mismatch": (ra[:80], [110.0, 105.0], 1.0, 1.0, False, 7, 256 * 100, "mismatched"),
        "reset_into_mismatch": (ra[:80], [110.0, 105.0], 0.5, 1.5, True, 8, 256 * 100, "matched"),
        "noisefree_mismatch": (ra[:120], [110.0, 105.0], 0.0, 1.5, True, 9, 256 * 120, None),
    }


def gen_single():
    lr.load()
    out = {"versions": versions()}
    for name, (acts, init, sig, a0, mism, zseed, zlen, prior) in single_env_cases().items():
        z = np.random.default_rng(zseed).standard_normal(zlen)
        env = lr.new_env()
        z_used = z
        if prior is not None:
            # run a short prior episode on the SAME env so simulator.is_mismatched is stale at reset
            zp = np.random.default_rng(100 + zseed).standard_normal(4096)
            lr.rollout(random_actions(5, seed=11), [105.0, 105.0], 1.0, 1.0, prior == "mismatched", zp, env=env)
        rec = lr.rollout(acts, init, sig, a0, mism, z_used, env=env)
        used = int(rec["cursor"][-1])
        out[f"{name}/actions"] = np.asarray(acts, dtype=np.float64)
        out[f"{name}/init"] = np.asarray(init)
        out[f"{name}/params"] = np.array([sig, a0, float(mism), float(prior == "mismatched")])
        out[f"{name}/z"] = z[:used + 8]
        for k in KEEP:
            out[f"{name}/{k}"] = rec[k]
        print(f"{name}: T={len(acts)} draws={used} max_attempts={rec['attempts'].max()} first_done="
              f"{int(np.argmax(rec['done'])) if rec['done'].any() else -1}")
    np.savez_compressed(os.path.join(GOLDEN_DIR, "single_env.npz"), **out)


def gen_batch(n_env=48, T=96, zlen_per=80 * 96):
    """SURVEY §8d C2 subset: float32-rounded inits ~U[100,120)^2 (default_rng(2)), per-env
    noise streams, per-env random actions; sigma in {0, 1} and one mismatched set."""
    lr.load()
    rng = np.random.default_rng(2)
    init = rng.uniform(100, 120, size=(n_env, 2)).astype(np.float32)
    arng = np.random.default_rng(12)
    acts = np.stack([arng.uniform(0, 20, size=(T, n_env)), arng.uniform(0, 2 * np.pi, size=(T, n_env))], axis=-1)
    z = np.random.default_rng(22).standard_normal((n_env, zlen_per))
    out = {"versions": versions(), "init": init, "actions": acts}
    used_max = 0
    for tag, (sig, a0, mism) in {"sigma0": (0.0, 1.0, False), "sigma1": (1.0, 1.0, False),
                                 "mismatch": (0.5, 1.5, True)}.items():
        recs = [lr.rollout(acts[:, e], init[e], sig, a0, mism, z[e]) for e in range(n_env)]
        out[f"{tag}/params"] = np.array([sig, a0, float(mism), 0.0])
        for k in KEEP:
            if k.startswith("reset_"):
                out[f"{tag}/{k}"] = np.stack([np.asarray(r[k]) for r in recs], axis=0)   # [n_env, ...]
            else:
                out[f"{tag}/{k}"] = np.stack([r[k] for r in recs], axis=1)               # [T, n_env, ...]
        used_max = max(used_max, max(int(r["cursor"][-1]) for r in recs))
        print(f"batch {tag}: draws max={max(int(r['cursor'][-1]) for r in recs)} "
              f"max_attempts={max(int(r['attempts'].max()) for r in recs)}")
    out["z"] = z[:, :used_max + 8]
    np.savez_compressed(os.path.join(GOLDEN_DIR, "batch_env.npz"), **out)


def gen_gp():
    """SURVEY §8d C4 at reduced size (N_train=300) through the reference's own LearningModule
    object: fixed-kernel sklearn GPRs installed on it, outputs of .error() and objective()."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, WhiteKernel

    mods = lr.load()
    LM = mods["Learning_module"]
    rng = np.random.default_rng(0)
    n = 300
    X = np.sort(rng.uniform(-np.pi, np.pi, n))
    yx = 0.2 + 0.5 * np.cos(X + 0.3) + 0.09 * rng.standard_normal(n)
    yy = -0.1 + 0.4 * np.sin(X - 0.2) + 0.09 * rng.standard_normal(n)
    lm = LM.LearningModule()
    lm.gprX = GaussianProcessRegressor(kernel=RBF(0.2) + WhiteKernel(0.008), optimizer=None)
    lm.gprY = GaussianProcessRegressor(kernel=RBF(0.25) + WhiteKernel(0.008), optimizer=None)
    lm.gprX.fit(X.reshape(-1, 1), yx)
    lm.gprY.fit(X.reshape(-1, 1), yy)
    lm.a0, lm.freq, lm.Dx, lm.Dy = 1.4, 4.0, 0.21, -0.12
    qrng = np.random.default_rng(5)
    vd = qrng.standard_normal((64, 2)) * 5
    err = np.array([np.concatenate(lm.error(v)) for v in vd])              # Learning_module.py:186-196
    alphas = qrng.uniform(-np.pi, np.pi, 64)
    obj = np.array([float(np.ravel(LM.objective(a, lm.a0, lm.freq, vd[i], lm.gprX, lm.gprY, lm.Dx, lm.Dy))[0])
                    for i, a in enumerate(alphas)])                         # Learning_module.py:10-24
    # LearningModule.predict (Learning_module.py:198-224): the bounded minimisation itself, live
    pred = np.array([np.concatenate([np.atleast_1d(np.asarray(o, dtype=float)).ravel() for o in lm.predict(v)]) for v in vd[:24]])
    q = np.linspace(-np.pi, np.pi, 257).reshape(-1, 1)
    mx, sx = lm.gprX.predict(q, return_std=True)
    my, sy = lm.gprY.predict(q, return_std=True)
    np.savez_compressed(
        os.path.join(GOLDEN_DIR, "gp.npz"), versions=versions(), X=X, yx=yx, yy=yy,
        lsx=0.2, lsy=0.25, noise=0.008, alpha_x=lm.gprX.alpha_, alpha_y=lm.gprY.alpha_,
        hyper=np.array([lm.a0, lm.freq, lm.Dx, lm.Dy]), vd=vd, error=err, predict=pred, obj_alpha=alphas, objective=obj,
        grid=q.ravel(), grid_mx=mx, grid_sx=sx, grid_my=my, grid_sy=sy)
    print("gp: error() rows", err.shape, "sigma range", err[:, 2].min(), err[:, 2].max())


def gen_learn():
    """main.py flow at reduced size through the reference's own run_sim + LearningModule: idle run ->
    estimateDisturbance, circle run -> learn().  Records the deterministic preprocessing outputs
    (Dx, Dy, a0, X, Yx, Yy); the GPR hyper-parameter search itself is sklearn's and not pinned."""
    mods = lr.load()
    LM, utils = mods["Learning_module"], mods["utils"]
    import contextlib, io
    freq, a0_def, dt, sigma = 4.0, 1.5, 0.030, 0.5
    idle = np.zeros((60, 3)); idle[:, 2] = np.arange(60) * dt
    T = 240
    circ = np.zeros((T, 3)); circ[:, 0] = freq; circ[:, 1] = np.linspace(-np.pi, np.pi, T); circ[:, 2] = np.arange(T) * dt
    z1 = np.random.default_rng(31).standard_normal(60 * 1500)
    z2 = np.random.default_rng(32).standard_normal(T * 1500)
    with contextlib.redirect_stdout(io.StringIO()):
        with lr.patched_noise(z1) as n1:
            px_i, py_i, _, t_i, _ = utils.run_sim(idle, init_pos=np.array([0, 0]), noise_var=sigma, a0=a0_def, is_mismatched=True)
            used1 = n1.cursor
        with lr.patched_noise(z2) as n2:
            px, py, al, tm, _ = utils.run_sim(circ, init_pos=np.array([0, 0]), noise_var=sigma, a0=a0_def, is_mismatched=True)
            used2 = n2.cursor
        lm = LM.LearningModule()
        lm.gprX.n_restarts_optimizer = 0
        lm.gprY.n_restarts_optimizer = 0
        lm.estimateDisturbance(px_i, py_i, t_i)
        a0 = lm.learn(px, py, al, tm.copy(), circ)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "learn.npz"), versions=versions(), idle=idle, circ=circ, z1=z1[:used1 + 8],
                        z2=z2[:used2 + 8], px_idle=px_i, py_idle=py_i, t_idle=t_i, px=px, py=py, alpha=al, time=tm,
                        Dx=lm.Dx, Dy=lm.Dy, a0=a0, X=lm.X, Yx=lm.Yx, Yy=lm.Yy, params=np.array([sigma, a0_def, freq]))
    print("learn: a0", a0, "D", lm.Dx, lm.Dy, "n", len(lm.X), "draws", used1, used2)


def gen_learn_fit():
    """The GPR fit itself, through the reference's LearningModule with its own settings (5 optimiser restarts,
    Learning_module.py:28-33,122-123) on the trajectory of learn.npz.  The restarts draw from numpy's global RandomState,
    seeded here; recorded: the fitted hyper-parameters, log marginal likelihoods, posterior on a grid and predict()."""
    mods = lr.load()
    LM = mods["Learning_module"]
    import contextlib, io
    g = np.load(os.path.join(GOLDEN_DIR, "learn.npz"))
    seed = 123
    with contextlib.redirect_stdout(io.StringIO()):
        lm = LM.LearningModule()
        lm.estimateDisturbance(g["px_idle"], g["py_idle"], g["t_idle"])
        np.random.seed(seed)
        a0 = lm.learn(g["px"].copy(), g["py"].copy(), g["alpha"].copy(), g["time"].copy(), g["circ"])
        grid = np.linspace(-3.0, 3.0, 97)
        mx, sx = lm.gprX.predict(grid.reshape(-1, 1), return_std=True)
        my, sy = lm.gprY.predict(grid.reshape(-1, 1), return_std=True)
        freq = g["circ"][0, 0]
        ang = np.linspace(0.1, 2 * np.pi - 0.1, 12)
        vd = a0 * freq * np.stack([np.cos(ang), np.sin(ang)], 1)
        pred = np.array([[float(np.ravel(v)[0]) for v in lm.predict(v_)] for v_ in vd])
    np.savez_compressed(os.path.join(GOLDEN_DIR, "learn_fit.npz"), versions=versions(), seed=seed, a0=a0,
                        theta_x=lm.gprX.kernel_.theta, theta_y=lm.gprY.kernel_.theta,
                        lml_x=lm.gprX.log_marginal_likelihood_value_, lml_y=lm.gprY.log_marginal_likelihood_value_,
                        grid=grid, grid_mx=mx, grid_sx=sx, grid_my=my, grid_sy=sy, vd=vd, predict=pred)
    print("learn_fit: theta", lm.gprX.kernel_.theta, lm.gprY.kernel_.theta, "lml", lm.gprX.log_marginal_likelihood_value_)


def gen_learn_2d():
    """Learning_module_2d.py through the reference's run_sim: idle run -> estimateDisturbance, a circle driven at a
    varying frequency (main_2d.py:149-158) -> learn(px, py, alpha, freq, time); then error() and predict()."""
    mods = lr.load()
    LM2, utils = lr.load_2d(), mods["utils"]
    import contextlib, io
    a0_def, dt, sigma = 1.5, 0.030, 0.3
    idle = np.zeros((60, 3)); idle[:, 2] = np.arange(60) * dt
    T = 300
    act = np.zeros((T, 3)); act[:, 1] = np.tile(np.linspace(-np.pi, np.pi, 100), 3)
    act[:, 0] = (np.cos(np.arange(T) / 5) + 1) / 2 * 4.9 + 0.1; act[:, 2] = np.arange(T) * dt
    z1 = np.random.default_rng(51).standard_normal(60 * 1500)
    z2 = np.random.default_rng(52).standard_normal(T * 1500)
    seed = 77
    with contextlib.redirect_stdout(io.StringIO()):
        with lr.patched_noise(z1):
            px_i, py_i, _, t_i, _ = utils.run_sim(idle, init_pos=np.array([0, 0]), noise_var=sigma, a0=a0_def, is_mismatched=True)
        with lr.patched_noise(z2):
            px, py, al, tm, fr = utils.run_sim(act, init_pos=np.array([0, 0]), noise_var=sigma, a0=a0_def, is_mismatched=True)
        lm = LM2.LearningModule()
        lm.estimateDisturbance(px_i, py_i, t_i)
        np.random.seed(seed)
        a0 = lm.learn(px.copy(), py.copy(), np.asarray(al, float).copy(), np.asarray(fr, float).copy(), np.asarray(tm, float).copy())
        lm.a0 = a0                                        # the reference's learn() returns a0 without storing it
        ang = np.linspace(-2.5, 2.5, 6)
        vd = np.stack([a0 * 2.5 * np.cos(ang), a0 * 2.5 * np.sin(ang)], 1)
        err = np.array([[float(np.ravel(v)[0]) for v in lm.error(v_)] for v_ in vd])
        pred = []
        for v_ in vd:
            X, mx, my, sx, sy = lm.predict(v_)
            pred.append([X[0], X[1], float(mx[0]), float(my[0]), float(sx[0]), float(sy[0])])
    np.savez_compressed(os.path.join(GOLDEN_DIR, "learn_2d.npz"), versions=versions(), seed=seed, px_idle=px_i, py_idle=py_i,
                        t_idle=t_i, px=px, py=py, alpha=np.asarray(al, float), freq=np.asarray(fr, float), time=np.asarray(tm, float),
                        Dx=lm.Dx, Dy=lm.Dy, a0=a0, X=lm.X, Yx=lm.Yx, Yy=lm.Yy, theta_x=lm.gprX.kernel_.theta,
                        theta_y=lm.gprY.kernel_.theta, lml_x=lm.gprX.log_marginal_likelihood_value_,
                        lml_y=lm.gprY.log_marginal_likelihood_value_, vd=vd, error=err, predict=np.array(pred))
    print("learn_2d: a0", a0, "theta", lm.gprX.kernel_.theta, lm.gprY.kernel_.theta, "n", len(lm.X))
    print("   predict", np.array(pred)[:2])


def gen_ddpg_host():
    """The two TensorFlow-free classes of RL/MR_ddpg.py run as they are: OUNoise on a fixed normal stream, and
    ReplayBuffer's ring / sampling behaviour (which transitions survive an overflow, batches without repeats)."""
    dd = lr.load_ddpg()
    z = np.random.default_rng(41).standard_normal(2 * 40)
    ou = dd.OUNoise(mu=np.zeros(2))
    with lr.patched_noise(z) as ns:
        xs = np.array([ou() for _ in range(40)])
        assert ns.cursor == 80
    rb = dd.ReplayBuffer(8, 0)
    for k in range(11):                                   # transition k: s = [k]*5, a = [k, -k], r = 10 + k, t = k % 3 == 0
        rb.add(np.full(5, float(k)), np.array([float(k), -float(k)]), 10.0 + k, k % 3 == 0, np.full(5, k + 0.5))
    kept = np.array([e[2] - 10.0 for e in rb.buffer])     # ids of the transitions still stored, oldest first
    s_b, a_b, r_b, t_b, s2_b = rb.sample_batch(4)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "ddpg_host.npz"), versions=versions(), ou_z=z, ou_x=xs,
                        ou_params=np.array([ou.theta, ou.sigma, ou.dt]), kept=kept, size=rb.size(),
                        batch_ids=r_b - 10.0, batch_s=s_b, batch_t=np.asarray(t_b, dtype=np.float64))
    print("ddpg_host: OU last", xs[-1], "kept", kept, "batch", r_b - 10.0)


def gen_recording(n_env=3, K=60, max_steps=12):
    """The reference's own transition logger (MR_data.MRExperiment) attached to the live MR_Env (MR_env.py:94-95,
    190-198) while a caller loop in the style of RL/MR_ddpg.py:268-311 resets on `done`: several episodes per env
    (time-outs at a shortened max_timesteps, one env that starts next to the goal).  Stored per env: the logger's
    per-episode arrays concatenated, the episode lengths, and every input (start positions per episode, actions,
    noise stream) so the device path can be fed the same run."""
    import contextlib
    import importlib
    import io
    import tempfile
    mods = lr.load()
    MRExperiment = importlib.import_module("MR_data").MRExperiment
    rng = np.random.default_rng(17)
    acts = np.stack([rng.uniform(0, 20, (K, n_env)), rng.uniform(0, 2 * np.pi, (K, n_env))], -1)
    E = K                                                     # more start positions than episodes can occur
    inits = rng.uniform(100, 120, (E, n_env, 2)).astype(np.float32).astype(np.float64)
    inits[1, 2] = [31.0, 5.0]                                 # env 2's second episode starts next to the goal radius
    acts[:, 2, 0] = 20.0; acts[:, 2, 1] = np.pi               # ... and drives towards it (x decreasing)
    zlen = 40 * K
    z = rng.standard_normal((zlen, n_env))
    out = {"actions": acts, "inits": inits, "z": z, "max_steps": max_steps, "versions": versions()}
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "_experiments"))
        os.chdir(tmp)
        try:
            for j in range(n_env):
                env = lr.new_env()
                env.max_timesteps = max_steps
                env.MR_data = MRExperiment()
                env.name_experiment = "golden"
                with lr.patched_noise(z[:, j]) as ns, contextlib.redirect_stdout(io.StringIO()):
                    ep = 0
                    # first episode starts at inits[-1] (the device run's explicit reset); later ones at inits[e - 1]
                    env.reset(init=inits[E - 1, j].copy(), noise_var=1, a0=1)
                    for k in range(K):
                        _, _, done, _ = env.step(acts[k, j])
                        if done and k < K - 1:
                            ep += 1
                            env.reset(init=inits[ep - 1, j].copy(), noise_var=1, a0=1)
                    out[f"env{j}/cursor"] = ns.cursor
                d = env.MR_data.__dict__
                n_ep = d["iterations"] + 1
                out[f"env{j}/steps"] = np.array([d["steps"][e] for e in range(n_ep)])
                for key in ("states", "observations", "actions", "rewards"):
                    out[f"env{j}/{key}"] = np.concatenate([np.asarray(d[key][e], dtype=np.float64).reshape(d["steps"][e] + 1, -1)
                                                           for e in range(n_ep)])
                print(f"recording: env {j}: {n_ep} episodes, lengths {out[f'env{j}/steps'].tolist()}, draws {ns.cursor}")
        finally:
            os.chdir(cwd)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "recording.npz"), **out)


def sweep_regime(seed):
    """Inputs of random regime `seed` (tests/test_live_reference_sweep.py): all drawn from default_rng(500 + seed)."""
    rng = np.random.default_rng(500 + seed)
    n, T = 6, 25
    scale = float(rng.choice([20.0, 150.0, 4000.0, 7000.0]))
    sigma = float(rng.choice([0.0, 0.02, 0.05] if scale < 100 else [0.0, 0.05, 0.5, 1.0]))
    a0 = float(rng.choice([0.5, 1.0, 1.5, 4.0]))
    mism = bool(rng.integers(0, 2))
    init = rng.uniform(-scale, scale, (n, 2))
    acts = np.stack([rng.uniform(-5, 30, (T, n)), rng.uniform(-7, 7, (T, n))], -1)
    acts[rng.random((T, n)) < 0.05] = 0.0
    z = rng.standard_normal((n, 200 * T + 64))
    return dict(n=n, T=T, sigma=sigma, a0=a0, mism=mism, init=init, acts=acts, z=z)


def sweep_reference(r):
    """Step every env of regime `r` through MR_Env: positions [T, n, 2], done [T, n], draws used [n].  The live
    reference when its tree is present, otherwise oracle/scipy_env.py — the reference's env restated on scipy's RK45,
    pinned to the live-reference goldens by tests/test_oracle_golden.py.  Returns the arrays and the source's name."""
    import contextlib
    import io
    from .scipy_env import ScipyEnv
    live = lr.available()
    pos, done, cursor = np.zeros((r["T"], r["n"], 2)), np.zeros((r["T"], r["n"]), np.uint8), np.zeros(r["n"], np.int64)
    for i in range(r["n"]):
        with contextlib.redirect_stdout(io.StringIO()), lr.patched_noise(r["z"][i]) as ns:
            env = lr.new_env() if live else ScipyEnv(normal=ns)
            env.reset(r["init"][i].copy(), noise_var=r["sigma"], a0=r["a0"], is_mismatched=r["mism"])
            for k in range(r["T"]):
                _, _, d, _ = env.step(r["acts"][k, i].copy())
                pos[k, i] = np.array(env.last_pos if live else env.y, dtype=np.float64)
                done[k, i] = bool(d)
            cursor[i] = ns.cursor
    return pos, done, cursor, "MR_RL MR_Env (live)" if live else "oracle/scipy_env.py on scipy RK45"


def gen_sweep(seeds=6):
    """The six random regimes of tests/test_live_reference_sweep.py (scale up to 7000, sigma up to 1, a0 in
    {0.5, 1, 1.5, 4}, mismatch on or off).  The inputs are regenerated from their seeds; stored are the positions,
    done flags and final noise cursors, and which implementation produced them."""
    out = {"versions": versions()}
    for seed in range(seeds):
        pos, done, cursor, source = sweep_reference(sweep_regime(seed))
        out[f"seed{seed}/pos"], out[f"seed{seed}/done"], out[f"seed{seed}/cursor"] = pos, done, cursor
    out["source"] = np.array(source)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "sweep.npz"), **out)


if __name__ == "__main__":
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    import sys
    if len(sys.argv) > 1:                                     # python -m oracle.gen_golden recording [...]
        for name in sys.argv[1:]:
            globals()["gen_" + name]()
        raise SystemExit(0)
    gen_single()
    gen_batch()
    gen_gp()
    gen_learn()
    gen_learn_fit()
    gen_learn_2d()
    gen_ddpg_host()
    gen_recording()
    gen_sweep()
