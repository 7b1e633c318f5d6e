"""MRExperiment wire format (MR_data.py) written from rollout arrays; checked against what the reference's own logger
recorded (tests/golden/recording.npz), and against the live logger where the reference tree is present."""
import contextlib
import io

import numpy as np
import pytest

from mr_rl_b200.recording import experiment_dict, load_experiment, save_experiment
from oracle import live_reference as lr
from oracle import mr_oracle as mo


def _oracle_run(T=40):
    rng = np.random.default_rng(4)
    acts = np.stack([rng.uniform(0, 20, T), rng.uniform(0, 2 * np.pi, T)], 1)
    z = rng.standard_normal(40 * T)
    r = mo.rollout(acts, [110.0, 105.0], 1.0, 1.0, False, z)
    return acts, z, r


def test_experiment_dict_structure_roundtrip(tmp_path):
    acts, z, r = _oracle_run()
    xy = r["pos"].T[None].transpose(2, 1, 0)                    # [K, 2, N=1]
    exp = experiment_dict([110.0, 105.0], acts, xy, done=r["done"][:, None])
    assert exp["iterations"] == 0 and exp["steps"][0] == len(acts)
    assert exp["states"][0].shape == (41, 2) and exp["observations"][0].shape == (41, 5)
    assert exp["actions"][0].shape == (41, 2) and exp["rewards"][0].shape == (41, 1)
    assert np.all(exp["actions"][0][0] == 0) and exp["rewards"][0][0, 0] == 0 and np.all(exp["rewards"][0][1:] == 10)
    assert np.allclose(exp["observations"][0][:, 4], np.hypot(*exp["states"][0].T))
    p = tmp_path / "exp.pickle"
    save_experiment(exp, p)
    back = load_experiment(p)
    assert set(back) == {"iterations", "states", "observations", "actions", "rewards", "steps", "info", "viewer",
                         "scream", "obs_states_str", "time_step"}
    assert np.array_equal(back["states"][0], exp["states"][0])


def test_wire_format_equals_the_reference_logger():
    """experiment_dict against what the reference's MRExperiment logger (MR_env.py:94-95,190-198) recorded: always the
    first episode of every env of the golden recording.npz, from the trajectory of the same inputs through the oracle;
    where the reference tree is present, also a live run with the logger attached, keys and scalars included."""
    g = _golden_recording()
    acts, inits, z, max_steps = g["actions"], g["inits"], g["z"], int(g["max_steps"])
    K, n_env = acts.shape[:2]
    E = inits.shape[0]
    xy, done = np.zeros((K, 2, n_env)), np.zeros((K, n_env), bool)
    for j in range(n_env):
        s = mo.SimState(noise=mo.NoiseCursor(z[:, j]))
        mo.env_reset(s, inits[E - 1, j], 1.0, 1.0, False)
        for k in range(K):
            obs, _, done[k, j] = mo.env_step(s, acts[k, j], max_steps=max_steps)[:3]
            xy[k, :, j] = obs[:2]
    mine = experiment_dict(inits[E - 1], acts, xy, done=done, until_done=True)
    assert mine["iterations"] == n_env - 1
    for j in range(n_env):
        n = int(g[f"env{j}/steps"][0])
        assert mine["steps"][j] == n, j
        for key in ("states", "observations", "actions", "rewards"):
            ref = g[f"env{j}/{key}"][:n + 1]
            assert mine[key][j].shape == ref.shape, (key, j)
            assert np.allclose(mine[key][j], ref, rtol=1e-9, atol=1e-12), (key, j)
    if not lr.available():
        return
    acts, z, r = _oracle_run()
    mods = lr.load()
    env = lr.new_env()
    import importlib
    MRExperiment = importlib.import_module("MR_data").MRExperiment
    env.MR_data = MRExperiment()
    env.name_experiment = "unused"
    with lr.patched_noise(z), contextlib.redirect_stdout(io.StringIO()):
        env.reset(init=np.array([110.0, 105.0]), noise_var=1.0, a0=1.0)
        for a in acts:
            env.step(a)
    ref = env.MR_data.__dict__
    xy = r["pos"].T[None].transpose(2, 1, 0)
    mine = experiment_dict([110.0, 105.0], acts, xy)
    assert set(mine) == set(ref)
    n = ref["steps"][0]
    assert n == len(acts)
    for key in ("states", "observations", "actions", "rewards"):
        a, b = np.asarray(ref[key][0], dtype=np.float64), mine[key][0][:n + 1]
        assert a.shape == b.shape, key
        assert np.allclose(a, b, rtol=1e-9, atol=1e-12), key
    assert mine["time_step"] == ref["time_step"] and mine["iterations"] == ref["iterations"]


@pytest.mark.gpu
def test_recorded_device_rollout_in_reference_format(tmp_path):
    import torch

    from mr_rl_b200 import VecMREnv
    n, K = 5, 60
    env = VecMREnv(n, device="cuda:0", noise="philox", seed=2)
    env.reset(init=np.array([110.0, 105.0]), noise_var=1.0, a0=1.0)
    rng = np.random.default_rng(0)
    acts = torch.as_tensor(np.stack([rng.uniform(0, 20, (K, n)), rng.uniform(0, 6.28, (K, n))], -1), device="cuda:0")
    res = env.rollout(actions=acts, record=True, record_done=True)
    exp = experiment_dict([110.0, 105.0], acts, res["xy"], done=res["done_traj"], until_done=True)
    assert exp["iterations"] == n - 1 and all(exp["steps"][e] == 51 for e in range(n))      # timeout at counter 51
    assert np.allclose(exp["states"][3][-1], res["xy"][50, :, 3].cpu().numpy())
    save_experiment(exp, tmp_path / "e")
    assert load_experiment(tmp_path / "e")["observations"][4].shape == (52, 5)


def test_logger_class_matches_array_builder():
    """MRExperiment (host logger with the reference's method names) fed step by step == experiment_dict."""
    from mr_rl_b200.recording import MRExperiment
    acts, z, r = _oracle_run(12)
    lg = MRExperiment()
    s0 = np.array([110.0, 105.0])
    lg.new_iter(s0, np.array([110.0, 105.0, 0, 0, np.hypot(110.0, 105.0)]), np.zeros(2), np.array([0]))
    for k in range(12):
        lg.new_transition(r["pos"][k], r["obs"][k], acts[k], 10)
    xy = r["pos"].T[None].transpose(2, 1, 0)
    ref = experiment_dict(s0, acts, xy)
    for key in ("states", "observations", "actions", "rewards"):
        assert np.allclose(np.asarray(lg.__dict__[key][0], dtype=float), ref[key][0])
    assert lg.steps[0] == 12 and set(lg.__dict__) == set(ref)


@pytest.mark.gpu
def test_mr_env_facade_logging_hook(tmp_path, monkeypatch):
    from mr_rl_b200 import MR_Env
    monkeypatch.chdir(tmp_path)
    env = MR_Env(device="cuda:0", noise="philox", seed=1)
    env.set_save_experice("unit")
    env.reset(init=np.array([110.0, 105.0]))
    for _ in range(5):
        env.step(np.array([10.0, 0.5]))
    d = env.MR_data
    assert d.iterations == 0 and d.steps[0] == 5 and d.observations[0].shape == (6, 5) and d.actions[0].shape == (6, 2)


def _golden_recording():
    import os
    from conftest import GOLDEN
    return np.load(os.path.join(GOLDEN, "recording.npz"))


def _check_against_reference_logger(exp, g, n_env):
    """exp: dict in the MRExperiment layout with env-major episode numbering; g: the golden of the reference's own logger."""
    it = 0
    for j in range(n_env):
        steps = g[f"env{j}/steps"]
        offs = np.concatenate([[0], np.cumsum(steps + 1)])
        for e, m in enumerate(steps):
            assert exp["steps"][it] == int(m), (j, e)
            for key in ("states", "observations", "actions", "rewards"):
                ref = g[f"env{j}/{key}"][offs[e]:offs[e + 1]]
                got = np.asarray(exp[key][it], dtype=np.float64)
                assert got.shape == ref.shape, (key, j, e, got.shape, ref.shape)
                assert np.allclose(got, ref, rtol=1e-9, atol=1e-12), (key, j, e)
            it += 1
    assert exp["iterations"] == it - 1


def test_vectorised_episode_flush_reproduces_the_reference_logger_on_oracle_data():
    """experiment_from_rollout (numpy index arithmetic, no loop over envs) fed with the per-step arrays the rollout kernel
    records — produced here by the scalar oracle with the same reset-on-done loop — must give exactly what the reference's
    MRExperiment logged in the live run (golden recording.npz: several episodes per env, a goal episode)."""
    from mr_rl_b200.recording import experiment_from_rollout
    g = _golden_recording()
    acts, inits, z, max_steps = g["actions"], g["inits"], g["z"], int(g["max_steps"])
    K, n_env = acts.shape[:2]
    E = inits.shape[0]
    res = {k: np.zeros(s) for k, s in (("xy", (K, 2, n_env)), ("done_traj", (K, n_env)), ("actions_traj", (K, n_env, 2)),
                                       ("rew_traj", (K, n_env)), ("reset_xy", (K, 2, n_env)), ("start_xy", (n_env, 2)))}
    for j in range(n_env):
        s = mo.SimState(noise=mo.NoiseCursor(z[:, j]))
        mo.env_reset(s, inits[E - 1, j], 1.0, 1.0, False)
        res["start_xy"][j] = inits[E - 1, j]
        ep = 0
        for k in range(K):
            obs, rew, done = mo.env_step(s, acts[k, j], max_steps=max_steps)[:3]
            res["xy"][k, :, j] = obs[:2]; res["done_traj"][k, j] = done; res["rew_traj"][k, j] = rew
            res["actions_traj"][k, j] = acts[k, j]
            if done and k < K - 1:
                ep += 1
                mo.env_reset(s, inits[ep - 1, j], 1.0, 1.0, False)
                res["reset_xy"][k, :, j] = inits[ep - 1, j]
        assert s.noise.cursor == int(g[f"env{j}/cursor"])
    _check_against_reference_logger(experiment_from_rollout(res), g, n_env)


@pytest.mark.gpu
def test_device_recorded_episodes_equal_the_reference_logger(tmp_path):
    """The same run on the device: ONE fused rollout launch with auto reset (start positions from the golden's list,
    table noise), per-episode keys written by the kernel, flushed to the MRExperiment layout — compared with what the
    reference's logger recorded in the live run, and round-tripped through the pickle."""
    import torch

    from mr_rl_b200 import VecMREnv, experiment_from_rollout
    g = _golden_recording()
    acts, inits, z, max_steps = g["actions"], g["inits"], g["z"], int(g["max_steps"])
    K, n_env = acts.shape[:2]
    E = inits.shape[0]
    env = VecMREnv(n_env, device="cuda:0", noise="table", noise_table=z, auto_reset=True)
    env.max_timesteps = max_steps
    env.reset(init=inits[E - 1], noise_var=1.0, a0=1.0)
    res = env.rollout(actions=torch.as_tensor(acts, device="cuda:0"), record_episodes=True, reset_init=inits)
    env.check_status()
    for j in range(n_env):
        assert int(env._cursor[j]) == int(g[f"env{j}/cursor"])
    exp = experiment_from_rollout(res)
    _check_against_reference_logger(exp, g, n_env)
    # the kernel's own keys agree with the split
    ep, st, dn = res["episode"].cpu().numpy(), res["step"].cpu().numpy(), res["done_traj"].cpu().numpy().astype(bool)
    for j in range(n_env):
        steps = g[f"env{j}/steps"]
        assert np.array_equal(ep[:, j], np.repeat(np.arange(len(steps)), steps))
        assert np.array_equal(st[:, j], np.concatenate([np.arange(1, m + 1) for m in steps]))
    assert np.array_equal(env._episode_counter.cpu().numpy(), dn.sum(0))
    save_experiment(exp, tmp_path / "rec")
    back = load_experiment(tmp_path / "rec")
    assert back["iterations"] == exp["iterations"] and np.array_equal(back["states"][2], exp["states"][2])
