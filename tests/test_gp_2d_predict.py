"""LearningModule2D.predict_batch / mr_gp_correct_action_2d: the corrected (alpha, f) of Learning_module_2d.py:239-268 for
a batch of desired velocities, solved on the device, against the reference's scipy search (LearningModule2D.predict) on
the same device model, and against the live reference's goldens (learn_2d.npz)."""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import Golden

LO, HI = np.array([-np.pi, 0.0]), np.array([np.pi, 5.0])
MAX_PASS = 64


@pytest.fixture(scope="module")
def g2():
    return Golden("learn_2d.npz")


# ---- numpy model of the problem (np.exp, independent of the kernel's table exponential) ----------------------------------
class Problem:
    """r(x) = a0 f (cos alpha, sin alpha) + (muX, muY)(x) - vd and g = J^T r from the fitted sklearn models' arrays."""

    def __init__(self, gx, gy, a0):
        self.a0 = float(a0)
        self.gps = [(g.X_train_ / g.kernel_.k1.length_scale, g.alpha_.ravel(), g.kernel_.k1.length_scale) for g in (gx, gy)]

    def _mean_grad(self, x, k):
        xs, al, ls = self.gps[k]
        s = x / ls - xs
        w = np.exp(-0.5 * (s * s).sum(1)) * al
        return w.sum(), -(w @ s) / ls

    def residual(self, x, vd):
        (mx, gx), (my, gy) = self._mean_grad(x, 0), self._mean_grad(x, 1)
        c, s = math.cos(x[0]), math.sin(x[0])
        af = self.a0 * x[1]
        r = np.array([af * c + mx - vd[0], af * s + my - vd[1]])
        J = np.array([[-af * s + gx[0], self.a0 * c + gx[1]], [af * c + gy[0], self.a0 * s + gy[1]]])
        return r, J.T @ r

    def F(self, x, vd):
        r, _ = self.residual(x, vd)
        return float(r @ r)

    def kkt(self, x, vd):
        """projected gradient |x - clip(x - J^T r)|_inf relative to 1 + |vd|^2"""
        _, g = self.residual(x, vd)
        return float(np.abs(x - np.clip(x - g, LO, HI)).max()) / (1.0 + float(vd @ vd))

    def start(self, vd):
        return np.clip([math.atan2(vd[1], vd[0]), math.hypot(vd[0], vd[1]) / self.a0], LO, HI)


def velocities(regime, n, a0, seed):
    """desired velocities a0 f_d (cos alpha_d, sin alpha_d) of one regime of the desired (alpha_d, f_d)"""
    rng = np.random.default_rng(seed)
    if regime == "interior":        # the minimum is a root inside the box
        ad, fd = rng.uniform(-np.pi + 0.5, np.pi - 0.5, n), rng.uniform(1.0, 3.5, n)
    elif regime == "f_upper":       # f ends on its upper bound
        ad, fd = rng.uniform(-np.pi, np.pi, n), rng.uniform(5.5, 7.0, n)
    elif regime == "alpha_pi":      # alpha_d within 0.25 of +-pi
        ad = np.where(rng.random(n) < 0.5, np.pi - rng.uniform(0, 0.25, n), -np.pi + rng.uniform(0, 0.25, n))
        fd = rng.uniform(0.5, 4.5, n)
    elif regime == "low":           # f_d < 0.5: the GP offset dominates, multimodal along alpha near f = 0
        ad, fd = rng.uniform(-np.pi, np.pi, n), rng.uniform(0.0, 0.5, n)
    else:
        raise ValueError(regime)
    return a0 * fd[:, None] * np.stack([np.cos(ad), np.sin(ad)], 1)


@pytest.fixture(scope="module")
def fixed():
    """The golden 2-D model at the golden theta (sklearn, optimizer=None: deterministic), installed on the device."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, WhiteKernel

    from mr_rl_b200.learning_module_2d import LearningModule2D
    g = Golden("learn_2d.npz")
    fit = lambda y, th: GaussianProcessRegressor(RBF(np.exp(th[0])) + WhiteKernel(np.exp(th[1])), optimizer=None).fit(g["X"], y)
    gx, gy = fit(g["Yx"], g["theta_x"]), fit(g["Yy"], g["theta_y"])
    lm = LearningModule2D(device="cuda:0", fit="host")
    lm.set_models(gx, gy, float(g["a0"]))
    assert lm._dx.n_train == 272 and lm._dx.n_pad == 384          # not a multiple of 128: the padding path
    return lm, Problem(gx, gy, g["a0"])


def solve(lm, vd):
    X, mx, my, sx, sy, it, st = lm.predict_batch(vd, return_info=True)
    return X.cpu().numpy(), it.cpu().numpy(), st.cpu().numpy()


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_action_2d_argument_errors_need_no_gpu():
    from mr_rl_b200 import _lib as L
    lib = L.load()
    D2 = C.c_double * 2

    def model(dim=2, n_train=272, n_pad=384, xs=8, al=8):
        return L.GPModel(xs, al, None, n_train, n_pad, dim, 0, 1.0, 0.1)

    gx, gy = model(), model()
    lo, hi = D2(-np.pi, 0.0), D2(np.pi, 5.0)
    P = 16                                                         # a fake device address: never dereferenced

    def call(gx=gx, gy=gy, vd=P, n=4, a0=1.9, lo=lo, hi=hi, x=P):
        rc = lib.mr_gp_correct_action_2d(C.byref(gx) if gx is not None else None, C.byref(gy) if gy is not None else None,
                                         vd, n, a0, lo, hi, x, None, None, None)
        return rc, lib.mr_last_error().decode()

    cases = [
        (dict(gx=None), -1, "null model"),
        (dict(gy=model(xs=None)), -1, "null model"),
        (dict(gx=model(al=None)), -1, "null model"),
        (dict(gx=model(dim=1)), -3, "dim 2"),
        (dict(gy=model(dim=1)), -3, "dim 2"),
        (dict(gy=model(n_train=271)), -1, "share"),
        (dict(gy=model(n_pad=512)), -1, "share"),
        (dict(n=-1), -1, "bad n"),
        (dict(vd=None), -1, "null vd"),
        (dict(x=None), -1, "x_out"),
        (dict(lo=D2(np.pi, 0.0)), -1, "lo < hi"),
        (dict(hi=D2(np.pi, -1.0)), -1, "lo < hi"),
        (dict(hi=D2(np.inf, 5.0)), -1, "finite"),
        (dict(lo=D2(-np.pi, np.nan)), -1, "finite"),
        (dict(a0=0.0), -1, "a0"),
        (dict(a0=-1.0), -1, "a0"),
        (dict(a0=np.nan), -1, "a0"),
        (dict(a0=np.inf), -1, "a0"),
    ]
    for kw, want, msg in cases:
        rc, err = call(**kw)
        assert rc == want and "mr_gp_correct_action_2d" in err and msg in err, (kw, rc, err)
    assert call(n=0, vd=None, x=None)[0] == 0                     # nothing to do: returns before any pointer is used


# ---- GPU -------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_action_2d_golden_velocities_match_reference_and_scipy(g2):
    import torch

    from conftest import rel_err
    from mr_rl_b200.learning_module_2d import LearningModule2D
    lm = LearningModule2D(device="cuda:0", fit="device")
    lm.estimateDisturbance(g2["px_idle"], g2["py_idle"], g2["t_idle"])
    np.random.seed(int(g2["seed"]))
    a0 = lm.learn(g2["px"], g2["py"], g2["alpha"], g2["freq"], g2["time"].copy())
    assert rel_err(a0, g2["a0"]) < 1e-12
    X, mx, my, sx, sy, it, st = lm.predict_batch(g2["vd"], return_info=True)
    assert X.shape == (6, 2) and X.dtype == torch.float64 and X.device.type == "cuda"
    assert (st == 0).all() and int(it.max()) <= 20
    Xh = X.cpu().numpy()
    for i, (vd, p_ref) in enumerate(zip(g2["vd"], g2["predict"])):
        # the bars test_2d_module_fit_error_predict_match_the_live_reference puts on predict()
        assert abs(np.angle(np.exp(1j * (Xh[i, 0] - p_ref[0])))) < 2e-2 and abs(Xh[i, 1] - p_ref[1]) < 2e-2
        ref_obj = lm._objective(p_ref[:2], vd)
        assert abs(lm._objective(Xh[i], vd) - ref_obj) < 1e-4 * (1 + abs(ref_obj))
        Xs, *_ = lm.predict(vd)                                    # the reference's scipy search on the same model
        assert np.abs(Xh[i] - Xs).max() <= 1e-4, (i, Xh[i], Xs)
    # the posterior is gp_batch at the minimiser: the same means bit for bit; the std kernel sums its column blocks with
    # shared-memory atomics, so repeated calls agree to rounding rather than bitwise
    mx2, my2, sx2, sy2 = lm.gp_batch(X)
    assert torch.equal(mx, mx2) and torch.equal(my, my2)
    assert float(((sx - sx2).abs() / sx2).max()) < 1e-13 and float(((sy - sy2).abs() / sy2).max()) < 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["interior", "f_upper", "alpha_pi"])
def test_action_2d_regimes_agree_with_scipy(fixed, regime):
    lm, pb = fixed
    vd = velocities(regime, 256, pb.a0, seed={"interior": 1, "f_upper": 2, "alpha_pi": 3}[regime])
    X, it, st = solve(lm, vd)
    assert (st == 0).all(), np.flatnonzero(st)
    for i in range(len(vd)):
        Xs, *_ = lm.predict(vd[i])
        assert np.abs(X[i] - Xs).max() <= 1e-4, (i, vd[i], X[i], Xs)
        assert pb.F(X[i], vd[i]) <= pb.F(Xs, vd[i]) + 1e-12
        if regime == "interior":                                   # the minimum is a root, solved to rounding
            assert math.sqrt(pb.F(X[i], vd[i])) <= 1e-9 * (1 + np.hypot(*vd[i]))
    # observed passes (B200): interior mean ~9 / max 18 in a numpy model of the solver; the bar leaves room
    bound = 24 if regime == "interior" else 32
    assert int(it.max()) <= bound, (regime, int(it.max()), float(it.mean()))
    print(f"{regime}: passes mean {it.mean():.1f} max {it.max()}")


@pytest.mark.gpu
def test_action_2d_low_speed_is_a_descent_to_a_kkt_point(fixed):
    lm, pb = fixed
    vd = np.vstack([np.zeros((1, 2)), velocities("low", 255, pb.a0, seed=4)])
    X, it, st = solve(lm, vd)
    assert (st == 0).all() and np.isfinite(X).all()
    assert np.array_equal(pb.start(vd[0]), [0.0, 0.0])
    agree = 0
    for i in range(len(vd)):
        assert pb.kkt(X[i], vd[i]) <= 1e-6, (i, vd[i], X[i])
        assert pb.F(X[i], vd[i]) <= pb.F(pb.start(vd[i]), vd[i])
        Xs, *_ = lm.predict(vd[i])
        agree += int(np.abs(X[i] - Xs).max() <= 1e-4)
    # multimodal along alpha on the f = 0 face: neither search is global, so agreement is reported, not asserted
    print(f"low speed: {agree}/{len(vd)} rows agree with scipy; passes mean {it.mean():.1f} max {it.max()}")


@pytest.mark.gpu
def test_action_2d_rows_are_batch_invariant_and_stay_in_bounds(fixed):
    import torch

    from mr_rl_b200 import _lib as L
    lm, pb = fixed
    vd = np.vstack([velocities(r, 1025, pb.a0, seed=10 + k) for k, r in enumerate(("interior", "f_upper", "alpha_pi", "low"))])
    vd = np.vstack([vd, [[0.0, 0.0]]])
    assert len(vd) == 4101
    vd = vd[:4097]
    Xb, itb, stb = solve(lm, vd)
    assert ((Xb >= LO) & (Xb <= HI)).all()
    for i in (0, 1, 1024, 1025, 2050, 3075, 4096):
        X1, it1, st1 = solve(lm, vd[i:i + 1])
        assert np.array_equal(X1[0].view(np.int64), Xb[i].view(np.int64)) and it1[0] == itb[i] and st1[0] == stb[i], i

    lib = L.load()
    lo, hi = (C.c_double * 2)(*LO), (C.c_double * 2)(*HI)
    for n in (1, 31, 33, 4097):
        pad = 67
        v = torch.as_tensor(vd[:n], device="cuda:0").contiguous()
        x = torch.full((n + pad, 2), 77.0, dtype=torch.float64, device="cuda:0")
        it = torch.full((n + pad,), 77, dtype=torch.int32, device="cuda:0")
        st = torch.full((n + pad,), 77, dtype=torch.uint8, device="cuda:0")
        rc = lib.mr_gp_correct_action_2d(C.byref(lm._dx._c), C.byref(lm._dy._c), v.data_ptr(), n, float(lm.a0), lo, hi,
                                         x.data_ptr(), it.data_ptr(), st.data_ptr(), None)
        assert rc == 0
        torch.cuda.synchronize()
        assert bool((x[n:] == 77).all()) and bool((it[n:] == 77).all()) and bool((st[n:] == 77).all()), n
        assert np.array_equal(x[:n].cpu().numpy(), Xb[:n]) and np.array_equal(it[:n].cpu().numpy(), itb[:n])


@pytest.mark.gpu
def test_action_2d_non_finite_rows_are_flagged_alone(fixed):
    import torch

    from mr_rl_b200 import _lib as L
    lm, pb = fixed
    good = velocities("interior", 5, pb.a0, seed=7)
    vd = good.copy()
    vd[1, 0] = np.nan
    vd[3, 1] = np.inf
    vd[4, 0] = -np.inf
    X, it, st = solve(lm, vd)
    Xg, itg, stg = solve(lm, good)
    assert list(st) == [0, 2, 0, 2, 2]
    assert np.isnan(X[[1, 3, 4]]).all()
    assert np.array_equal(X[[0, 2]], Xg[[0, 2]]) and np.array_equal(it[[0, 2]], itg[[0, 2]])
    # n = 0: nothing to launch, nothing written
    out = lm.predict_batch(np.zeros((0, 2)), return_info=True)
    assert all(t.shape[0] == 0 for t in out)
    lib = L.load()
    assert lib.mr_gp_correct_action_2d(C.byref(lm._dx._c), C.byref(lm._dy._c), None, 0, 1.0, (C.c_double * 2)(*LO),
                                       (C.c_double * 2)(*HI), None, None, None, None) == 0
    torch.cuda.synchronize()
