"""The C oracle stepped through random regimes against MR_Env on the same noise streams — pins the oracle beyond the
fixed regimes of the other golden vectors.  Always against tests/golden/sweep.npz (written by
oracle/gen_golden.py:gen_sweep, which names its source in the file); in addition against the UNMODIFIED reference
(MR_Env behind import stubs) where its tree is present."""
import contextlib
import io
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import live_reference as lr
from oracle.gen_golden import sweep_regime


@pytest.fixture(scope="module")
def golden_sweep():
    return np.load(os.path.join(GOLDEN, "sweep.npz"))


@pytest.mark.parametrize("seed", range(6))
def test_c_oracle_equals_the_live_reference_in_random_regimes(seed, golden_sweep):
    from oracle import c_oracle
    r = sweep_regime(seed)
    n, T, z = r["n"], r["T"], r["z"]
    ref = c_oracle.rollout(r["init"], r["acts"], r["sigma"], r["a0"], mism=r["mism"], mism_at_reset=False, z=z)
    assert ref["bad"] == 0
    g = {k: golden_sweep[f"seed{seed}/{k}"] for k in ("pos", "done", "cursor")}
    assert np.array_equal(ref["done"], g["done"]), seed
    assert np.array_equal(ref["cursor"], g["cursor"]), seed
    for i in range(n):
        err = np.abs(g["pos"][:, i] - ref["pos"][:, i]).max() / max(1.0, np.abs(ref["pos"][:, i]).max())
        assert err < 1e-12, (seed, i, err)
    if not lr.available():
        return
    for i in range(n):
        env = lr.new_env()
        with contextlib.redirect_stdout(io.StringIO()), lr.patched_noise(z[i]) as ns:
            env.reset(r["init"][i].copy(), noise_var=r["sigma"], a0=r["a0"], is_mismatched=r["mism"])
            pos, done = [], []
            for k in range(T):
                _, _, d, _ = env.step(r["acts"][k, i].copy())
                pos.append(np.array(env.last_pos, dtype=np.float64).copy()); done.append(bool(d))
            cursor = ns.cursor
        assert done == [bool(v) for v in ref["done"][:, i]], (seed, i)
        assert cursor == int(ref["cursor"][i])
        err = np.abs(np.array(pos) - ref["pos"][:, i]).max() / max(1.0, np.abs(ref["pos"][:, i]).max())
        assert err < 1e-12, (seed, i, err)
