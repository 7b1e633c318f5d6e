"""mr_gp_predict (csrc/mr_gp.cu) on every launch path, against an extended-precision reference.

The entry point picks one of five code paths:
  - staged K_q / mean (gp_kq_mean_smem_kernel): the model fits in shared memory and x_train_scaled, alpha are
    16-byte aligned;
  - global K_q / mean (gp_kq_mean_kernel): otherwise (dim 1 from n_pad 12 800, dim 2 from n_pad 8 576, or an
    unaligned model);
  - triangular std (gp_var_kernel, dense = 0, and gp_std_finish_kernel) in chunks of 16 384 queries, proj_rows == 0;
  - fused spectral mean and std (gp_posterior_spectral_kernel<DIM, NT>), proj_rows > 0;
  - two-kernel spectral std (gp_var_kernel, dense = 1), with MR_GP_FUSED=0 (read once per process).

The models are built directly as mr_gp_model structs: the C contract accepts any scaled inputs, alpha, triangular
linv or dense projection whose padding is zero, so a synthetic model can sit on either side of every selection
boundary without a large Cholesky factorisation.  One model per dimension from DeviceGP.fit ties them to real use.

The reference runs in np.longdouble (80-bit on x86-64).  It reproduces the device's float64 input rounding, so that
in dim 1 the exponent is the device's own argument x = -0.5 fl(fl(fl(q / l) - x_j)^2), and only the exponential and
the sums are compared.  Every bound is derived from the operation (see reference()).
"""
import ctypes as C
import math
import os
import re
import subprocess
import sys
from decimal import Decimal, localcontext

import numpy as np
import pytest
import torch

from mr_rl_b200 import _lib as L

LD = np.longdouble
U = 2.0 ** -53                       # unit roundoff of float64
U_EXP = 2.0 ** -51                   # 2 ulp of the exponential, relative (ulp(y) <= 2^-52 |y|)
U_REF = 2.0 ** -63                   # unit roundoff of the reference, twice over
GUARD = 64                           # sentinel elements behind every output and the workspace
SENTINEL = 7.25e300
CHUNK = 16384                        # kGpChunk: queries per pass of the triangular std pipeline
SMEM_LIMIT = 200 * 1024              # launch_kq_mean: the staged kernel's shared-memory cap
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gamma(n):
    """Higham's gamma_n = n u / (1 - n u): the relative error bound of a sum of depth n in float64."""
    return n * U / (1.0 - n * U)


# ---- models -------------------------------------------------------------------------------------------------------------
class HostModel:
    """The arrays of one mr_gp_model on the host.  W is the triangular L^-1 (proj_rows == 0) or the dense projection
    (proj_rows > 0) in row-sorted COO form without duplicates, every row below n_rows holding at least one entry."""

    def __init__(self, X, alpha, ls, noise, n_pad=None, W=None, proj_rows=0):
        X = np.asarray(X, dtype=np.float64)
        self.n_train, self.dim = X.shape
        self.n_pad = n_pad or (self.n_train + L.GP_PAD - 1) // L.GP_PAD * L.GP_PAD
        self.ls, self.noise = float(ls), float(noise)
        self.diag = np.float64(1.0) + np.float64(noise)              # what the host passes the kernels
        self.xs = np.zeros((self.n_pad, self.dim))
        self.xs[:self.n_train] = X / self.ls                          # as DeviceGP scales them: a query on a training
        self.alpha = np.zeros(self.n_pad)                             # point gives fl(q / l) == x_j, k = 1 exactly
        self.alpha[:self.n_train] = alpha
        self.W, self.proj_rows = W, proj_rows


def lower_w(rng, n_train, n_pad, nnz_row, diag, frac=0.8, clip=True):
    """A random lower-triangular W with the diagonal and up to nnz_row - 1 further entries per row, scaled so that
    |W k|^2 <= sum_r (sum_c |W_rc|)^2 = frac (1 + noise) for every k in [0, 1]^n.  With clip, the diagonal entry of
    the last row is 3 sqrt(1 + noise): a query on the last training point then has |W k|^2 > 4 (1 + noise) and the
    variance is clipped to 0."""
    r = np.repeat(np.arange(n_train), nnz_row - 1)
    c = np.floor(rng.random(r.size) * r).astype(np.int64)           # c < r (row 0 keeps only its diagonal)
    keys = np.unique(np.concatenate([r * n_pad + c, np.arange(n_train) * (n_pad + 1)]))
    return _scaled_coo(rng, keys // n_pad, keys % n_pad, n_train, n_pad, diag, frac, clip)


def dense_p(rng, proj_rows, n_train, n_pad, diag, frac=0.8, clip=True):
    """A dense [proj_rows][n_pad] projection with zero padding columns, scaled as lower_w; with clip, P[0][n_train-1]
    = 3 sqrt(1 + noise)."""
    r, c = np.divmod(np.arange(proj_rows * n_train), n_train)
    return _scaled_coo(rng, r, c, proj_rows, n_pad, diag, frac, clip, clip_at=(0, n_train - 1))


def _scaled_coo(rng, r, c, n_rows, n_pad, diag, frac, clip, clip_at=None):
    v = rng.standard_normal(r.size)
    ptr = np.searchsorted(r, np.arange(n_rows))
    rowabs = np.add.reduceat(np.abs(v), ptr)
    v *= math.sqrt(frac * diag / float((rowabs ** 2).sum()))
    if clip:
        cr, cc = clip_at if clip_at else (n_rows - 1, n_rows - 1)
        v[np.flatnonzero((r == cr) & (c == cc))[0]] = 3.0 * math.sqrt(diag)
    return dict(rows=r, cols=c, vals=v, ptr=ptr, n_rows=n_rows)


class DeviceModel:
    """HostModel on the device as an mr_gp_model; misalign places x_train_scaled and / or alpha 8 bytes into a larger
    buffer, which makes them 8- but not 16-byte aligned."""

    def __init__(self, h, misalign=(), dev="cuda:0"):
        self.h = h
        self._keep = []

        def place(a, key):
            a = np.ascontiguousarray(a, dtype=np.float64).ravel()
            off = 1 if key in misalign else 0
            buf = torch.zeros(a.size + 2, dtype=torch.float64, device=dev)
            buf[off:off + a.size] = torch.from_numpy(a).to(dev)
            self._keep.append(buf)
            assert buf.data_ptr() % 16 == 0
            return buf, buf.data_ptr() + 8 * off, (buf, off, a)

        _, xp, self._x = place(h.xs, "x")
        _, ap, self._a = place(h.alpha, "alpha")
        self.Wd, wp = None, None
        if h.W is not None:
            rows = h.proj_rows if h.proj_rows else h.n_pad
            self.Wd = torch.zeros((rows, h.n_pad), dtype=torch.float64, device=dev)
            w = h.W
            self._wi = (torch.from_numpy(w["rows"]).to(dev), torch.from_numpy(w["cols"]).to(dev))
            self._wv = torch.from_numpy(w["vals"]).to(dev)
            self.Wd[self._wi] = self._wv
            wp = self.Wd.data_ptr()
        self.c = L.GPModel(xp, ap, wp, h.n_train, h.n_pad, h.dim, h.proj_rows, h.ls, h.noise)
        self.aligned = "x" not in misalign and "alpha" not in misalign

    def kq_path(self):
        """The K_q / mean kernel launch_kq_mean selects for this model."""
        smem = self.h.n_pad * (self.h.dim + 1) * 8 + 64 * 8 + 16
        return "staged" if smem <= SMEM_LIMIT and self.aligned else "global"

    def assert_unchanged(self):
        for buf, off, a in (self._x, self._a):
            got = buf.cpu().numpy()
            assert np.array_equal(got[off:off + a.size].view(np.int64), a.view(np.int64))
            assert not got[:off].any() and not got[off + a.size:].any()
        if self.Wd is not None:
            assert int(torch.count_nonzero(self.Wd)) == self.h.W["vals"].size
            assert torch.equal(self.Wd[self._wi], self._wv)


# ---- the device call --------------------------------------------------------------------------------------------------
def predict(m, q, want_std=True, lib=None):
    """mr_gp_predict with sentinels behind mean, std and the workspace; asserts that none of them was written and that
    the model's buffers are unchanged."""
    lib = lib or L.load()
    q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, m.h.dim)
    n = len(q)
    dev = m.Wd.device if m.Wd is not None else m._keep[0].device
    qd = torch.from_numpy(q).to(dev)
    mean = torch.full((n + GUARD,), SENTINEL, dtype=torch.float64, device=dev)
    std = torch.full((n + GUARD,), SENTINEL, dtype=torch.float64, device=dev) if want_std else None
    ws_bytes = int(lib.mr_gp_workspace_bytes(C.byref(m.c), n, 1)) if want_std else 0
    assert ws_bytes % 8 == 0
    ws = torch.full((ws_bytes // 8 + GUARD,), SENTINEL, dtype=torch.float64, device=dev) if want_std else None
    rc = lib.mr_gp_predict(C.byref(m.c), qd.data_ptr(), n, mean.data_ptr(), std.data_ptr() if want_std else None,
                           ws.data_ptr() if want_std else None, ws_bytes, None)
    assert rc == 0, lib.mr_last_error().decode()
    torch.cuda.synchronize()
    assert bool((mean[n:] == SENTINEL).all()), "mean written past n_q"
    if want_std:
        assert bool((std[n:] == SENTINEL).all()), "std written past n_q"
        assert bool((ws[ws_bytes // 8:] == SENTINEL).all()), "workspace written past mr_gp_workspace_bytes"
    m.assert_unchanged()
    return mean[:n].cpu().numpy(), (std[:n].cpu().numpy() if want_std else None)


def mean_depth(path, n_pad):
    """Longest chain of roundings in one mean: the K_q kernels let each lane sum n_pad / 32 terms and add the 32 lanes
    in 5 shuffle levels; the fused spectral kernel lets each thread sum half a row, n_pad / 2 terms, plus one shuffle."""
    return n_pad // 2 + 1 if path == "spectral" else n_pad // 32 + 5


# ---- the reference ----------------------------------------------------------------------------------------------------
def reference(h, q, path, want_std=True):
    """Mean and variance in long double, with bounds on what the device may differ from them.

    Exponent.  In dim 1 the reference forms x_j = -0.5 fl(d_j^2), d_j = fl(fl(q / l) - x_j), as every kernel does, so
    k_j = exp(x_j) is the exact value of the device's own argument.  In dim 2 the staged and spectral kernels form
    fl(d1^2 + fl(d0^2)) with an fma, and the global kernel lets the compiler contract d0^2 + d1^2 as it likes; each
    is within 2 u d^2 of the exact d0^2 + d1^2 the reference uses, so k_j moves by at most |x_j| 2^-52 (relative,
    to first order; the factor 1.001 covers the rest).

    Mean.  The device k_j is k_j (1 + e_j) with |e_j| <= e = 2^-51 + [dim 2] 1.001 |x_j| 2^-52 (2 ulp of the
    exponential), and e = 1 below x = -707, where exp_neg_tab flushes to 0 and the library exp returns subnormals.
    Each term alpha_j k_j enters one fma chain and a shuffle tree of total depth D (mean_depth), so by
    the standard bound on recursive summation the computed mean is sum_j alpha_j k_j (1 + e_j)(1 + t_j), |t_j| <=
    gamma_D:
        |mean_dev - mean| <= sum_j |alpha_j k_j| ((1 + e)(1 + gamma_D) - 1).
    Padding columns meet alpha = 0 and zero columns of W and add exact zeros.

    Std.  V_r = sum_c W_rc k_c is one DMMA accumulation of at most n_pad products, so with A_r = sum_c |W_rc| k_c and
    B_r = sum_c |W_rc| k_c ((1 + e_c)(1 + gamma_{n_pad + 1}) - 1), |V_dev - V| <= B_r and |V_dev^2 - V^2| <= 2 A_r B_r
    + B_r^2.  The squares of the R rows (n_pad, or proj_rows) are summed in registers, shuffles and atomics of depth
    at most R + 8: |ssq_dev - ssq| <= E = sum_r (2 A_r B_r + B_r^2) + gamma_{R+8} sum_r (A_r + B_r)^2.  Then
    v = fl(diag - ssq_dev) and std = fl(sqrt(max(v, 0))) add one rounding each, std^2 two more:
        |std_dev^2 - max(diag - ssq, 0)| <= E + 3.01 u (|diag - ssq| + E).
    The clip to 0 is 1-Lipschitz, so the bound holds across it.  diag = fl(1 + noise) is the device's own argument.

    Reference error.  The long-double sums of n terms are within n 2^-64 of exact, covered by U_REF (n + 2) on the
    same absolute sums."""
    assert np.finfo(LD).nmant >= 63, "the reference needs an extended-precision long double"
    q = np.asarray(q, dtype=np.float64).reshape(-1, h.dim)
    assert np.isfinite(q).all()
    n, n_pad = h.n_train, h.n_pad
    xs, al = h.xs[:n], h.alpha[:n].astype(LD)
    g_mean = LD(gamma(mean_depth(path, n_pad)))
    out = dict(mean=[], mean_tol=[], v=[], v_tol=[], x=[])
    W = h.W
    block = max(1, min(64, int(3e6 // max(n_pad, W["vals"].size if want_std else 0))))
    if want_std:
        Wv, Wa = W["vals"].astype(LD), np.abs(W["vals"]).astype(LD)
        R = h.proj_rows if h.proj_rows else n_pad
        g_v, g_r = LD(gamma(n_pad + 1)), LD(gamma(R + 8))
    for b in range(0, len(q), block):
        qs = q[b:b + block] / h.ls
        d = qs[:, None, :] - xs[None, :, :]
        if h.dim == 1:
            x = (-0.5 * (d[..., 0] * d[..., 0])).astype(LD)
            e = np.full(x.shape, LD(U_EXP))
        else:
            dl = d.astype(LD)
            x = -0.5 * (dl * dl).sum(-1)
            e = LD(U_EXP) + LD(1.001 * 2.0 ** -52) * np.abs(x)
        e[x < -707.0] = 1                                           # flushed (exp_neg_tab) or subnormal (exp): any
        k = np.exp(x)                                               # value in [0, 2 k_j] is within the bound
        t = k * al
        at = np.abs(t)
        out["mean"].append(t.sum(1))
        out["mean_tol"].append((at * ((1 + e) * (1 + g_mean) - 1)).sum(1) + at.sum(1) * LD(U_REF * (n + 2)))
        out["x"].append(x.min(1))
        if want_std:
            kc = k[:, W["cols"]]
            V = np.add.reduceat(kc * Wv, W["ptr"], axis=1)
            A = np.add.reduceat(kc * Wa, W["ptr"], axis=1)
            B = np.add.reduceat(kc * ((1 + e[:, W["cols"]]) * (1 + g_v) - 1) * Wa, W["ptr"], axis=1)
            ssq = (V * V).sum(1)
            E = (2 * A * B + B * B).sum(1) + g_r * ((A + B) ** 2).sum(1) + ((A * A).sum(1)) * LD(U_REF * (n + R + 4))
            v = LD(h.diag) - ssq
            out["v"].append(v)
            out["v_tol"].append(E + LD(3.01 * U) * (np.abs(v) + E))
    return {k: np.concatenate(v) if v else None for k, v in out.items()}


def check(h, q, path, mean, std=None, rows=None):
    """mean (and std) of the device against reference(); rows restricts the check to a subset of the queries.
    Returns the largest error / bound ratios, for the record."""
    q = np.asarray(q, dtype=np.float64).reshape(-1, h.dim)
    idx = np.arange(len(q)) if rows is None else np.asarray(rows)
    ref = reference(h, q[idx], path, want_std=std is not None)
    em = np.abs(mean[idx].astype(LD) - ref["mean"])
    bad = np.flatnonzero(~(em <= ref["mean_tol"]))
    assert bad.size == 0, (path, "mean", idx[bad[:5]], mean[idx][bad[:5]], ref["mean"][bad[:5]], ref["mean_tol"][bad[:5]])
    worst = dict(mean=float((em / np.maximum(ref["mean_tol"], LD(1e-300))).max()))
    if std is not None:
        s2 = std[idx].astype(LD) ** 2
        ev = np.abs(s2 - np.maximum(ref["v"], 0))
        bad = np.flatnonzero(~(ev <= ref["v_tol"]))
        assert bad.size == 0, (path, "std", idx[bad[:5]], std[idx][bad[:5]], ref["v"][bad[:5]], ref["v_tol"][bad[:5]])
        clipped = ref["v"] < -ref["v_tol"]
        assert (std[idx][clipped] == 0).all()
        worst["std"] = float((ev / np.maximum(ref["v_tol"], LD(1e-300))).max())
        worst["clipped"] = int(clipped.sum())
    return worst


# ---- model factories ----------------------------------------------------------------------------------------------------
def synthetic(dim, n_train, n_pad=None, seed=0, ls=None, noise=0.05, std="tri", proj_rows=0, nnz_row=48, clip=True):
    """Training inputs over the heading range (dim 1) or the (alpha, f) box (dim 2), random alpha_, and a synthetic
    triangular W or dense projection."""
    rng = np.random.default_rng(seed)
    if dim == 1:
        X = np.sort(rng.uniform(-np.pi, np.pi, (n_train, 1)), axis=0)
    else:
        X = np.stack([rng.uniform(-np.pi, np.pi, n_train), rng.uniform(0.0, 5.0, n_train)], 1)
    ls = ls or (0.2 if dim == 1 else 0.6)
    alpha = 0.3 * rng.standard_normal(n_train)
    h = HostModel(X, alpha, ls, noise, n_pad=n_pad)
    if std == "tri":
        h.W = lower_w(rng, n_train, h.n_pad, nnz_row, h.diag, clip=clip)
    elif std == "proj":
        h.W, h.proj_rows = dense_p(rng, proj_rows, n_train, h.n_pad, h.diag, clip=clip), proj_rows
    return h, X


def queries(X, n, seed, with_training_points=True):
    """n queries over 1.1 times the training range, the first ones exactly on training points (k = 1), the last
    training point included (the clipped variance)."""
    rng = np.random.default_rng(seed)
    lo, hi = X.min(0), X.max(0)
    mid, half = (lo + hi) / 2, (hi - lo) / 2 * 1.1
    q = mid + half * rng.uniform(-1, 1, (n, X.shape[1]))
    if with_training_points and n >= 3:
        q[:3] = X[[0, len(X) // 2, len(X) - 1]]
    return q


@pytest.fixture(scope="module")
def lib():
    return L.load()


# ---- CPU: the exponential's constants and the argument checks ---------------------------------------------------------
def test_exp_range_reduction_constants_are_ln2_over_64():
    """exp_neg_tab reduces x by n ln2/64 as hi + lo in two fma steps.  hi must be short enough that n hi has no
    rounding for |n| < 2^17, and lo must be the correctly rounded rest of ln2/64 - hi: a shorter lo leaves every
    result too small by ~3.3e-17 |x| relative, 200 ulp at x = -700.  64/ln2 must be the float64 nearest to it."""
    src = open(os.path.join(ROOT, "mr_rl_b200", "csrc", "mr_gp.cu")).read()
    body = src[src.index("double exp_neg_tab("):]
    body = body[:body.index("\n}\n")]
    inv = re.search(r"x \* ([0-9.]+);", body).group(1)
    hi_s, lo_s = re.findall(r"fma\(-nd, (0x[0-9a-fp.+-]+), ", body)
    hi, lo = float.fromhex(hi_s), float.fromhex(lo_s)
    with localcontext() as ctx:
        ctx.prec = 60
        c = Decimal(2).ln() / 64
        rest = c - Decimal(hi)
    assert float(inv) == float(1 / c)
    m, _ = math.frexp(hi)
    mant = int(m * 2 ** 53)
    assert 53 - ((mant & -mant).bit_length() - 1) <= 36             # n hi exact for |n| < 2^17
    assert lo == float(rest), (lo.hex(), float(rest).hex())        # within half an ulp of lo, 2^-99, of ln2/64 - hi


def test_predict_argument_errors_need_no_gpu(lib):
    """Every check mr_gp_predict makes before a launch, each with its own message; none of them touches memory."""
    P = 1 << 20                                                    # fake, 16-byte aligned device addresses: never read

    def model(xs=P, al=P, linv=P, n_train=200, n_pad=256, dim=1, proj=0, ls=0.5):
        return L.GPModel(xs, al, linv, n_train, n_pad, dim, proj, ls, 0.1)

    def call(m="default", q=P, n=16, mean=P, std=P, ws=P, ws_bytes=1 << 40):
        m = model() if m == "default" else m
        rc = lib.mr_gp_predict(C.byref(m) if m is not None else None, q, n, mean, std, ws, ws_bytes, None)
        return rc, lib.mr_last_error().decode()

    need = int(lib.mr_gp_workspace_bytes(C.byref(model()), 16, 1))
    assert need == 128 * 256 * 8 + 128 * 8
    assert lib.mr_gp_workspace_bytes(C.byref(model()), 16, 0) == 0 and lib.mr_gp_workspace_bytes(C.byref(model()), 0, 1) == 0
    assert lib.mr_gp_workspace_bytes(C.byref(model()), 3 * CHUNK + 5, 1) == CHUNK * 256 * 8 + CHUNK * 8
    cases = [
        (dict(m=None), -1, "null model"),
        (dict(m=model(xs=None)), -1, "null model"),
        (dict(m=model(al=None)), -1, "null model"),
        (dict(n=-1), -1, "bad n_q"),
        (dict(q=None), -1, "null q/mean"),
        (dict(mean=None), -1, "null q/mean"),
        (dict(m=model(dim=3)), -3, "dim must be 1 or 2"),
        (dict(m=model(dim=0)), -3, "dim must be 1 or 2"),
        (dict(m=model(n_pad=200)), -1, "n_pad must be a positive multiple of 128"),
        (dict(m=model(n_pad=-128)), -1, "n_pad must be a positive multiple of 128"),
        (dict(m=model(n_train=0)), -1, "1 <= n_train <= n_pad"),
        (dict(m=model(n_train=257)), -1, "1 <= n_train <= n_pad"),
        (dict(m=model(ls=0.0)), -1, "bad length_scale"),
        (dict(m=model(ls=-0.5)), -1, "bad length_scale"),
        (dict(m=model(ls=float("nan"))), -1, "bad length_scale"),
        (dict(m=model(linv=None)), -1, "no linv"),
        (dict(m=model(proj=16)), -1, "proj_rows must be"),
        (dict(m=model(proj=-32)), -1, "proj_rows must be"),
        (dict(m=model(proj=160)), -1, "proj_rows must be"),
        (dict(m=model(proj=384)), -1, "proj_rows must be"),          # > n_pad
        (dict(m=model(proj=128, linv=P + 8)), -1, "projection must be 16-byte aligned"),
        (dict(ws=None), -1, "workspace too small"),
        (dict(ws_bytes=need - 8), -1, f"workspace too small ({need - 8} < {need})"),
        (dict(ws=P + 8), -1, "workspace must be 16-byte aligned"),
        (dict(m=model(linv=P + 8)), -1, "linv must be 16-byte aligned"),
    ]
    for kw, want, msg in cases:
        rc, err = call(**kw)
        assert rc == want and err.startswith("mr_gp_predict: ") and msg in err, (kw, rc, err)
    msgs = {call(**kw)[1].split(" (")[0] for kw, _, _ in cases}
    assert len(msgs) == 13                                         # one message per check
    # nothing to do: returns before any pointer is used
    assert call(n=0, q=None, mean=None, std=None, ws=None, ws_bytes=0)[0] == 0
    assert call(m=model(dim=3, linv=None), n=0)[0] == 0


# ---- GPU: the exponential at ulp level ------------------------------------------------------------------------------------
def exp_sweep():
    """Exponents over [-745, 0], uniform and log-spaced, x = 0, both sides of the flush threshold, and below -745.
    The queries are q = sqrt(-2 x); the exponent is then x = -0.5 fl(q^2), recomputed from q."""
    rng = np.random.default_rng(11)
    x = np.concatenate([-745.0 * rng.random(20000), -np.logspace(-30, np.log10(745.0), 20000), [0.0],
                        -rng.uniform(745.0, 1e4, 64)])
    q = np.sqrt(-2.0 * x)
    # the flush threshold: n = rint(x 64 / ln 2) = -65344.5 ... on a grid of ulp steps of q around it
    qt = math.sqrt(2.0 * 65344.5 * math.log(2) / 64)
    q = np.concatenate([q, qt + np.arange(-256, 257) * math.ulp(qt) * 1024])
    return q


def ulp_errors(got, x):
    """(got - exp(x)) in ulps of exp(x), ulps of subnormals included."""
    y = np.exp(x.astype(LD))
    _, e = np.frexp(y)
    ulp = np.maximum(np.ldexp(LD(1), (e - 53).astype(np.int32)), LD(2.0 ** -1074))
    return (got.astype(LD) - y) / ulp


RANGES = [(-1.0, 0.0), (-40.0, -1.0), (-200.0, -40.0), (-700.0, -200.0), (-745.0, -700.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["staged", "global", "spectral"])
def test_exponential_is_within_2_ulp(path):
    """n_train = 1, x_0 = 0, alpha = 1, l = 1: the mean is exactly exp_neg_tab(-0.5 fl(q^2)) on the staged and fused
    spectral paths, and the library exp of the same argument on the global path.  At most 2 ulp wherever the result
    is not flushed; exactly 0 where exp_neg_tab flushes (2^m T[j] p with m < -1021); exactly 1 at x = 0."""
    h = HostModel(np.zeros((1, 1)), [1.0], 1.0, 0.1)
    if path == "spectral":
        h.W, h.proj_rows = dense_p(np.random.default_rng(0), 32, 1, 128, h.diag, clip=False), 32
    m = DeviceModel(h, misalign=("alpha",) if path == "global" else ())
    assert path == "spectral" or m.kq_path() == path
    q = exp_sweep()
    mean, _ = predict(m, q, want_std=path == "spectral")
    x = -0.5 * (q * q)
    assert mean[np.flatnonzero(q == 0)[0]] == 1.0
    if path == "global":
        flushed = np.zeros(len(x), bool)
    else:
        n = np.rint(x * 92.33248261689366)
        flushed = np.floor(n / 64) < -1021
        assert flushed.any() and (~flushed & (x < -707)).any()        # both sides of the threshold were swept
        assert (mean[flushed] == 0).all(), x[flushed & (mean != 0)][:5]
    err = ulp_errors(mean, x)
    live = ~flushed
    report = []
    for a, b in RANGES:
        sel = live & (x >= a) & (x <= b)
        if sel.any():
            report.append(f"[{a:g}, {b:g}]: max {float(np.abs(err[sel]).max()):.2f} mean {float(err[sel].mean()):+.2f}")
    print(f"\n{path} exp ulp errors: " + "; ".join(report))
    worst = np.flatnonzero(~(np.abs(err) <= 2) & live)
    assert worst.size == 0, (path, report, x[worst[:5]], err[worst[:5]])


# ---- GPU: the selection boundaries of the K_q kernel ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dim,n_pad,path", [(1, 12672, "staged"), (1, 12800, "global"), (2, 8448, "staged"),
                                            (2, 8576, "global")])
def test_kq_kernel_selection_boundary(dim, n_pad, path):
    """On both sides of n_pad (dim + 1) 8 + 528 <= 200 KiB: the mean of 1 500 queries and the triangular std of 40,
    with a sparse synthetic L^-1 that touches every column block of the contraction."""
    h, X = synthetic(dim, n_pad - 37, n_pad, seed=n_pad, nnz_row=24)
    m = DeviceModel(h)
    assert m.kq_path() == path
    q = queries(X, 1500, seed=dim)
    mean, _ = predict(m, q, want_std=False)
    print(path, dim, n_pad, check(h, q, path, mean))
    mean2, std = predict(m, q[:40])
    assert np.array_equal(mean2.view(np.int64), mean[:40].view(np.int64))
    w = check(h, q[:40], path, mean2, std)
    assert w["clipped"] >= 1 and std[2] == 0                       # on the last training point
    print(path, dim, n_pad, "std", w)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2])
@pytest.mark.parametrize("misalign", [("x",), ("alpha",), ("x", "alpha")])
def test_unaligned_model_takes_the_global_kernel(dim, misalign):
    """x_train_scaled and / or alpha 8 bytes into their buffers: no TMA bulk copy is possible, so a small model runs
    the global K_q kernel, with the same results to within the bounds."""
    h, X = synthetic(dim, 300, seed=5 + dim)
    m, ma = DeviceModel(h, misalign=misalign), DeviceModel(h)
    assert m.kq_path() == "global" and ma.kq_path() == "staged"
    q = queries(X, 700, seed=dim)
    mean, std = predict(m, q)
    check(h, q, "global", mean, std)
    mean_a, std_a = predict(ma, q)
    check(h, q, "staged", mean_a, std_a)


# ---- GPU: the chunk loop of the triangular std ------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small_models():
    return {dim: synthetic(dim, 200, seed=20 + dim, nnz_row=64) for dim in (1, 2)}


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2])
@pytest.mark.parametrize("n_q", [1, 127, 128, 129, CHUNK - 1, CHUNK, CHUNK + 1, 3 * CHUNK + 5])
def test_chunk_loop(small_models, dim, n_q):
    """The std pipeline runs in chunks of 16 384 queries, each padded to a multiple of 128 rows.  Every mean is
    checked; the std on the rows around every chunk and tile edge and on a random sample."""
    h, X = small_models[dim]
    m = DeviceModel(h)
    q = queries(X, n_q, seed=n_q)
    mean, std = predict(m, q)
    check(h, q, "staged", mean, None)
    edges = {0, n_q - 1} | {e + o for e in range(0, n_q + 1, 128) for o in (-1, 0)} if n_q <= 256 else \
        {0, n_q - 1} | {c + o for c in range(0, n_q + 1, CHUNK) for o in (-2, -1, 0, 1, 127, 128)}
    rows = sorted(i for i in edges if 0 <= i < n_q)
    rows += list(np.random.default_rng(n_q).choice(n_q, min(n_q, 48), replace=False))
    check(h, q, "staged", mean, std, rows=np.unique(rows))


# ---- GPU: the fused spectral kernel ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2])
@pytest.mark.parametrize("proj_rows", [32, 64, 96, 128, 256, 384])
def test_fused_spectral_kernel(dim, proj_rows):
    """proj_rows 32 / 64 / 96 / 128+ select NT = 1 / 2 / 3 / 4 column tiles per warp; 256 and 384 take two and three
    128-row passes, and only the first accumulates the mean.  Ragged n_q: the last CTA is partly empty."""
    h, X = synthetic(dim, 450, seed=proj_rows + dim, std="proj", proj_rows=proj_rows)
    m = DeviceModel(h)
    q = queries(X, 300, seed=proj_rows)
    mean, std = predict(m, q)
    w = check(h, q, "spectral", mean, std)
    assert w["clipped"] >= 1
    mean_only, _ = predict(m, q, want_std=False)                   # the staged kernel: another summation order
    check(h, q, "staged", mean_only)


# ---- GPU: the two-kernel spectral path (MR_GP_FUSED=0) ------------------------------------------------------------------------
_TWO_KERNEL = r"""
import ctypes as C, sys
import numpy as np, torch
sys.path.insert(0, sys.argv[3])
from mr_rl_b200 import _lib as L
lib = L.load()
z = np.load(sys.argv[1])
out = {}
for i, R in enumerate(z["rows"]):
    xs, al, P, q = (torch.from_numpy(z[k]).cuda() for k in ("xs", "alpha", f"P{R}", "q"))
    m = L.GPModel(xs.data_ptr(), al.data_ptr(), P.data_ptr(), int(z["n_train"]), xs.shape[0], xs.shape[1], int(R),
                  float(z["ls"]), float(z["noise"]))
    n = q.shape[0]
    mean = torch.full((n + 64,), 7.25e300, dtype=torch.float64, device="cuda")
    std = mean.clone()
    wsb = int(lib.mr_gp_workspace_bytes(C.byref(m), n, 1))
    ws = torch.full((wsb // 8 + 64,), 7.25e300, dtype=torch.float64, device="cuda")
    rc = lib.mr_gp_predict(C.byref(m), q.data_ptr(), n, mean.data_ptr(), std.data_ptr(), ws.data_ptr(), wsb, None)
    torch.cuda.synchronize()
    out[f"rc{R}"] = np.array([rc])
    out[f"err{R}"] = np.array([lib.mr_last_error().decode()])
    out[f"mean{R}"], out[f"std{R}"] = mean.cpu().numpy(), std.cpu().numpy()
    out[f"ws{R}"] = ws[wsb // 8:].cpu().numpy()
    out[f"P{R}"] = P.cpu().numpy()
np.savez(sys.argv[2], **out)
"""


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2])
def test_two_kernel_spectral_path(tmp_path, dim):
    """MR_GP_FUSED=0 (read once per process, hence a subprocess) keeps the K_q kernel + gp_var_kernel(dense = 1) for the
    spectral form: proj_rows 128 and 256 agree with the reference, non-finite rows stay in their rows, and 96 is
    refused with MR_ERR_UNSUPPORTED, since that path contracts whole 128-row blocks."""
    rows = (128, 256, 96)
    hs, X = {}, None
    arrays = {}
    for R in rows:
        h, X = synthetic(dim, 450, seed=70 + dim, std="proj", proj_rows=R)
        hs[R] = h
        P = np.zeros((R, h.n_pad))
        P[h.W["rows"], h.W["cols"]] = h.W["vals"]
        arrays[f"P{R}"] = P
    h = hs[128]
    q = queries(X, 300, seed=dim)
    bad = q.copy()
    bad[7, 0], bad[100, dim - 1], bad[200] = np.nan, np.inf, -np.inf
    np.savez(tmp_path / "in.npz", xs=h.xs, alpha=h.alpha, q=bad, rows=np.array(rows), n_train=h.n_train, ls=h.ls,
             noise=h.noise, **arrays)
    env = dict(os.environ, MR_GP_FUSED="0")
    subprocess.run([sys.executable, "-c", _TWO_KERNEL, str(tmp_path / "in.npz"), str(tmp_path / "out.npz"), ROOT],
                   check=True, env=env, timeout=600)
    z = np.load(tmp_path / "out.npz")
    assert int(z["rc96"][0]) == -3 and "two-kernel path needs proj_rows in multiples of 128" in str(z["err96"][0])
    n = len(q)
    fin = np.setdiff1d(np.arange(n), [7, 100, 200])
    for R in (128, 256):
        assert int(z[f"rc{R}"][0]) == 0, str(z[f"err{R}"][0])
        mean, std = z[f"mean{R}"], z[f"std{R}"]
        assert (mean[n:] == SENTINEL).all() and (std[n:] == SENTINEL).all() and (z[f"ws{R}"] == SENTINEL).all()
        assert np.array_equal(z[f"P{R}"], arrays[f"P{R}"])
        w = check(hs[R], q, "staged", mean[:n], std[:n], rows=fin)
        assert w["clipped"] >= 1
        assert np.isnan(mean[7]) and np.isnan(std[7])
        assert mean[100] == 0 and mean[200] == 0 and std[100] == std[200] == np.sqrt(hs[R].diag)


# ---- GPU: training-set edges -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", ["staged", "global", "spectral"])
@pytest.mark.parametrize("n_train", [1, 127, 128, 129])
@pytest.mark.parametrize("regime", ["mixed", "underflow", "flat"])
def test_training_set_edges(path, n_train, regime):
    """n_train around one 128-column tile.  mixed: l = 0.2 with queries on training points (k = 1) and clipped
    variances; underflow: l = 1e-3 on inputs 0.05 apart, so almost every k underflows to 0 (or flushes); flat: l = 1e3,
    every k = 1 - O(1e-5) and alpha alternating in sign, so the mean is a cancelling sum and its bound scales with
    sum |alpha_j k_j| rather than with the mean."""
    rng = np.random.default_rng(n_train)
    ls = {"mixed": 0.2, "underflow": 1e-3, "flat": 1e3}[regime]
    X = np.sort(rng.uniform(-np.pi, np.pi, (n_train, 1)), axis=0) if regime != "underflow" else \
        (0.05 * np.arange(n_train) - 3.0).reshape(-1, 1)
    alpha = rng.standard_normal(n_train) if regime != "flat" else np.where(np.arange(n_train) % 2 == 0, 1.0, -1.0)
    h = HostModel(X, alpha, ls, 0.01)
    clip = regime == "mixed"
    if path == "spectral":
        h.W, h.proj_rows = dense_p(rng, 64, n_train, h.n_pad, h.diag, clip=clip), 64
    else:
        h.W = lower_w(rng, n_train, h.n_pad, 32, h.diag, clip=clip)
    m = DeviceModel(h, misalign=("x",) if path == "global" else ())
    assert path == "spectral" or m.kq_path() == path
    q = queries(X, 257, seed=n_train)
    if regime == "underflow":
        q[3:] = X[rng.integers(0, n_train, 254)] + rng.choice([0.0, 2e-3, 1e-2, 0.025], (254, 1))
    mean, std = predict(m, q)
    w = check(h, q, path, mean, std)
    assert (mean[:3] != 0).all()
    if regime == "mixed" and n_train > 1:
        assert w["clipped"] >= 1 and std[2] == 0                   # the last training point
    if regime == "flat" and n_train > 1:
        assert np.abs(mean).max() < 0.5 * np.abs(alpha).sum()       # the sum does cancel


# ---- GPU: non-finite queries ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2])
@pytest.mark.parametrize("path", ["staged", "global", "spectral"])
def test_non_finite_queries_stay_in_their_rows(dim, path):
    """A NaN query gives NaN mean and std in its own row only; a +-inf query has every k = 0, so mean exactly 0 and std
    exactly sqrt(1 + noise); the finite rows are what they are without the bad rows."""
    kw = dict(std="proj", proj_rows=128) if path == "spectral" else {}
    h, X = synthetic(dim, 300, seed=90 + dim, **kw)
    m = DeviceModel(h, misalign=("alpha",) if path == "global" else ())
    q = queries(X, 520, seed=dim)
    bad = q.copy()
    nan_rows, inf_rows = [5, 130, 519], [0, 131, 256, 400]
    bad[5, 0] = bad[130, dim - 1] = bad[519] = np.nan
    bad[0, 0], bad[131, dim - 1], bad[256] = np.inf, -np.inf, np.inf
    bad[400] = [np.inf, -np.inf][:dim]
    mean, std = predict(m, bad)
    assert np.isnan(mean[nan_rows]).all() and np.isnan(std[nan_rows]).all()
    assert (mean[inf_rows] == 0).all() and (std[inf_rows] == np.sqrt(h.diag)).all()
    fin = np.setdiff1d(np.arange(len(q)), nan_rows + inf_rows)
    assert np.isfinite(mean[fin]).all() and np.isfinite(std[fin]).all()
    clean, _ = predict(m, q[fin], want_std=False)
    if path != "spectral":
        assert np.array_equal(mean[fin].view(np.int64), clean.view(np.int64))
    check(h, q, path, mean, std, rows=fin)
    mo, _ = predict(m, bad, want_std=False)                        # the mean-only launch
    assert np.isnan(mo[nan_rows]).all() and (mo[inf_rows] == 0).all() and np.isfinite(mo[fin]).all()


# ---- GPU: reproducibility -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2])
@pytest.mark.parametrize("path", ["staged", "global", "spectral"])
def test_mean_is_bitwise_reproducible(dim, path):
    """A row's mean does not depend on the call, on n_q or on the row's position in the batch, and on the K_q kernels it
    is the same in the mean-only launch and in the launch that also computes the std.  The std sums with atomics, so it
    is only held to its bound."""
    kw = dict(std="proj", proj_rows=96) if path == "spectral" else {}
    h, X = synthetic(dim, 333, seed=40 + dim, **kw)
    m = DeviceModel(h, misalign=("x", "alpha") if path == "global" else ())
    q = queries(X, 1000, seed=dim)
    bits = lambda a: a.view(np.int64)
    full, std = predict(m, q)
    again, std2 = predict(m, q)
    assert np.array_equal(bits(full), bits(again))
    check(h, q, path, full, std)
    check(h, q, path, again, std2)
    if path != "spectral":
        mo, _ = predict(m, q, want_std=False)
        assert np.array_equal(bits(mo), bits(full))
    for sl in (slice(0, 1), slice(999, 1000), slice(137, 1000), slice(5, 42), slice(None, None, -1)):
        part, _ = predict(m, q[sl], want_std=path == "spectral")
        assert np.array_equal(bits(part), bits(full[sl])), sl
    tiled, _ = predict(m, np.concatenate([q, q, q[:300]]))
    assert np.array_equal(bits(tiled), bits(np.concatenate([full, full, full[:300]])))


# ---- GPU: models fitted by DeviceGP.fit ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2])
def test_fitted_model_every_path(dim):
    """A model from DeviceGP.fit (L^-1 with cancelling entries, the variance close to the noise floor near the data):
    triangular std, mean only, the same arrays unaligned (global kernel), and the spectral projection when
    enable_spectral_variance takes it."""
    from mr_rl_b200 import DeviceGP
    rng = np.random.default_rng(dim)
    n = 400
    if dim == 1:
        X = np.sort(rng.uniform(-np.pi, np.pi, (n, 1)), axis=0)
        y = 0.2 + 0.5 * np.cos(X[:, 0] + 0.3) + 0.09 * rng.standard_normal(n)
        ls = 0.25
    else:
        X = np.stack([rng.uniform(-np.pi, np.pi, n), rng.uniform(0.0, 5.0, n)], 1)
        y = 0.3 * np.sin(X[:, 0]) * X[:, 1] + 0.05 * rng.standard_normal(n)
        ls = 0.8
    gp = DeviceGP.fit(X, y, ls, 0.008, device="cuda:0")
    h = HostModel(X, gp._alpha.cpu().numpy()[:n], ls, 0.008, n_pad=gp.n_pad)
    h.xs = gp._xs.cpu().numpy()                                   # the device's own scaling of the inputs
    Wd = gp._linv.cpu().numpy()
    r, c = np.nonzero(Wd)
    h.W = dict(rows=r, cols=c, vals=Wd[r, c], ptr=np.searchsorted(r, np.arange(n)), n_rows=n)
    q = queries(X, 600, seed=dim)
    for misalign, path in (((), "staged"), (("alpha",), "global")):
        m = DeviceModel(h, misalign=misalign)
        assert m.kq_path() == path
        mean, std = predict(m, q)
        print(dim, path, check(h, q, path, mean, std))
        mo, _ = predict(m, q, want_std=False)
        assert np.array_equal(mo.view(np.int64), mean.view(np.int64))
    rows = gp.enable_spectral_variance()
    if dim == 1:
        assert rows > 0
    if rows:
        P = gp._proj.cpu().numpy()
        r, c = np.nonzero(P)
        hp = HostModel(X, h.alpha[:n], ls, 0.008, n_pad=gp.n_pad)
        hp.xs = h.xs
        hp.W, hp.proj_rows = dict(rows=r, cols=c, vals=P[r, c], ptr=np.searchsorted(r, np.arange(rows)), n_rows=rows), rows
        mp, sp = predict(DeviceModel(hp), q)
        print(dim, "spectral", rows, check(hp, q, "spectral", mp, sp))
