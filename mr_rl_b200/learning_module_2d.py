"""``LearningModule`` of Learning_module_2d.py: the disturbance GPs over (heading alpha, frequency f).

Same method surface as the reference's 2-D variant (estimateDisturbance, learn(px, py, alpha, freq, time), error,
predict; attrs gprX, gprY, X, Yx, Yy, a0, Dx, Dy).  The GPR fit (sklearn's search with 5 restarts, objective on the
device) and every GP evaluation run on the GPU with input dimension 2 (csrc/mr_gpfit.cu, csrc/mr_gp.cu); predict()
keeps the reference's scipy ``minimize`` over (alpha, f) with the bounds of Learning_module_2d.py:258, its objective
evaluated through the device GPs.  Preprocessing is the numpy/scipy restatement (per-frame frequencies, O(n)).
"""
from __future__ import annotations

import math

import numpy as np
import torch

from .gp import DeviceGP


class LearningModule2D:
    BOUNDS = ((-np.pi, np.pi), (0, 5))     # the (alpha, f) box of the corrected action, Learning_module_2d.py:258

    def __init__(self, device="cuda", fit="device"):
        if fit == "device":
            from .gpr import DeviceGPR
            self.gprX = DeviceGPR(n_restarts_optimizer=5, device=device)      # Learning_module_2d.py:29-33
            self.gprY = DeviceGPR(n_restarts_optimizer=5, device=device)
        elif fit == "host":
            from sklearn.gaussian_process import GaussianProcessRegressor
            from sklearn.gaussian_process.kernels import RBF, WhiteKernel
            kernel = RBF(length_scale=1.0, length_scale_bounds=(1e-2, 10.0)) + WhiteKernel()
            self.gprX = GaussianProcessRegressor(kernel=kernel, n_restarts_optimizer=5)
            self.gprY = GaussianProcessRegressor(kernel=kernel, n_restarts_optimizer=5)
        else:
            raise ValueError("fit must be 'device' or 'host'")
        self.device = device
        self.X, self.Yx, self.Yy = [], [], []
        self.a0 = 0
        self.f = 0
        self.Dx = 0
        self.Dy = 0
        self._dx = self._dy = None

    @staticmethod
    def _velocities(px, py, time):
        from scipy.ndimage import uniform_filter1d
        N = int(1 / 0.035 / 2)                                   # Learning_module_2d.py:48,70
        px = uniform_filter1d(px, N, mode="nearest")
        py = uniform_filter1d(py, N, mode="nearest")
        vx = uniform_filter1d(np.gradient(px, time), int(N / 2), mode="nearest")
        vy = uniform_filter1d(np.gradient(py, time), int(N / 2), mode="nearest")
        return N, vx, vy

    def estimateDisturbance(self, px, py, time):
        """Learning_module_2d.py:47-61: unlike the 1-D module the mean runs over ALL frames."""
        _, vx, vy = self._velocities(np.asarray(px, float), np.asarray(py, float), np.asarray(time, float))
        self.Dx = np.mean(vx)
        self.Dy = np.mean(vy)

    def _targets(self, px, py, alpha, freq, time):
        """learn() up to the fit (Learning_module_2d.py:65-120): a0, GP inputs X = (alpha, f) and residual targets."""
        time = np.asarray(time, float) - time[0]
        N, vx, vy = self._velocities(np.asarray(px, float), np.asarray(py, float), time)
        speed = np.sqrt((vx - self.Dx) ** 2 + (vy - self.Dy) ** 2)
        alpha, freq = np.asarray(alpha, float), np.asarray(freq, float)
        off = np.argwhere(alpha >= 500)                          # controller-off frames, :86-97
        if len(off) > 0:
            cut = int(off[0]) - 1
            alpha, freq, vx, vy, speed = alpha[:cut], freq[:cut], vx[:cut], vy[:cut], speed[:cut]
        alpha, freq, vx, vy, speed = alpha[N:-N], freq[N:-N], vx[N:-N], vy[N:-N], speed[N:-N]
        a0 = np.median(speed / freq)
        X = np.vstack([alpha, freq]).transpose()
        Yx = vx - a0 * freq * np.cos(alpha)
        Yy = vy - a0 * freq * np.sin(alpha)
        return a0, X, Yx, Yy

    def learn(self, px, py, alpha, freq, time):
        """Learning_module_2d.py:65-141.  alpha, freq: per-frame arrays.  Returns a0."""
        a0, X, Yx, Yy = self._targets(px, py, alpha, freq, time)
        self.gprX.fit(X, Yx)
        self.gprY.fit(X, Yy)
        self.X, self.Yx, self.Yy = X, Yx, Yy
        self.a0 = a0
        self.upload()
        return a0

    def upload(self):
        as_device = lambda g: g.device_model() if hasattr(g, "device_model") else DeviceGP.from_sklearn(g, self.device)
        self._dx = as_device(self.gprX)
        self._dy = as_device(self.gprY)
        self._dx.enable_spectral_variance()             # verified against the triangular form before it is used
        self._dy.enable_spectral_variance()

    def set_models(self, gprX, gprY, a0, Dx=0.0, Dy=0.0):
        self.gprX, self.gprY, self.a0, self.Dx, self.Dy = gprX, gprY, a0, Dx, Dy
        self.X = gprX.X_train_
        self.upload()

    # ---- device inference ----------------------------------------------------------------------------------------
    def gp_batch(self, X, return_std=True):
        """Posterior of both GPs at X [N, 2] = (alpha, f) -> (muX, muY[, sigX, sigY]) device tensors."""
        X = torch.as_tensor(X, dtype=torch.float64, device=self.device).reshape(-1, 2)
        if return_std:
            mx, sx = self._dx.predict(X, True)
            my, sy = self._dy.predict(X, True)
            return mx, my, sx, sy
        return self._dx.predict(X), self._dy.predict(X)

    def _desired(self, vd):
        vd = np.asarray(vd, float).ravel()
        return np.array([math.atan2(vd[1], vd[0]), np.linalg.norm(vd) / self.a0])      # :229-230

    def error(self, vd):
        """Learning_module_2d.py:226-237."""
        mx, my, sx, sy = (t.cpu().numpy() for t in self.gp_batch(self._desired(vd)))
        return mx, my, sx, sy

    def _objective(self, X, vd):
        """objective of Learning_module_2d.py:11-25 (no drift terms in the 2-D module)."""
        alpha, freq = float(X[0]), float(X[1])
        mx, my = self.gp_batch(np.array([alpha, freq]), False)
        mux, muy = float(mx[0]), float(my[0])
        a0 = self.a0
        return (a0 * freq) ** 2 + (mux - vd[0]) ** 2 + 2 * a0 * freq * np.cos(alpha) * (mux - vd[0]) \
            + (muy - vd[1]) ** 2 + 2 * a0 * freq * np.sin(alpha) * (muy - vd[1])

    def predict_batch(self, vd, return_info=False):
        """LearningModule2D.predict for vd [N, 2] (array or device tensor) in one device call (mr_gp_correct_action_2d):
        the minimiser over (alpha, f) in BOUNDS of the reference's objective, which equals |r|^2 for
        r = a0 f (cos alpha, sin alpha) + (muX, muY)(alpha, f) - vd, found by a projected Newton / Levenberg-Marquardt
        search with both GP means, gradients and Hessians evaluated on the device; then the posterior at the minimiser
        through gp_batch, the kernels error() uses.
        Returns (X [N, 2], muX, muY, sigX, sigY) device tensors, plus (iters [N] int32 passes, status [N] uint8) with
        ``return_info=True``.  Rows whose search did not converge are returned, not raised: status 1 = the 64-pass cap
        was reached and X is the best point found; status 2 = vd was not finite (or the GP means were not finite at the
        start point) and X is NaN."""
        import ctypes as C

        from . import _lib as L
        dev = torch.device(self.device)
        vd = torch.as_tensor(vd).to(device=dev, dtype=torch.float64).reshape(-1, 2).contiguous()
        n = vd.shape[0]
        X = torch.empty((n, 2), dtype=torch.float64, device=dev)
        iters = torch.empty(n, dtype=torch.int32, device=dev)
        status = torch.empty(n, dtype=torch.uint8, device=dev)
        (lo0, hi0), (lo1, hi1) = self.BOUNDS
        with torch.cuda.device(dev):
            rc = L.load().mr_gp_correct_action_2d(C.byref(self._dx._c), C.byref(self._dy._c), vd.data_ptr(), n, float(self.a0),
                                                  (C.c_double * 2)(lo0, lo1), (C.c_double * 2)(hi0, hi1), X.data_ptr(),
                                                  iters.data_ptr(), status.data_ptr(),
                                                  C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        L.check(rc, "mr_gp_correct_action_2d")
        mx, my, sx, sy = self.gp_batch(X)
        return (X, mx, my, sx, sy, iters, status) if return_info else (X, mx, my, sx, sy)

    def predict(self, vd):
        """Learning_module_2d.py:239-268: scipy minimize over (alpha, f) in [-pi, pi] x [0, 5] from the desired values."""
        from scipy.optimize import minimize
        vd = np.asarray(vd, float).ravel()
        x0 = self._desired(vd)
        result = minimize(self._objective, x0, args=(vd,), bounds=self.BOUNDS)
        X = np.array(result.x)
        mx, my, sx, sy = (t.cpu().numpy() for t in self.gp_batch(X))
        return X, mx, my, sx, sy
