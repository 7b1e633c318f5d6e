"""``LearningModule`` (Learning_module.py:27-224) with GP inference on the device.

Same attribute / method surface as the reference (gprX, gprY, X, Yx, Yy, a0, freq, Dx, Dy;
estimateDisturbance, learn, error, predict) plus batched entry points for the vectorised
control loop.  ``fit="device"`` (default) runs the GPR fit on the GPU too (gpr.DeviceGPR: sklearn's L-BFGS-B
search with 5 restarts, each objective evaluation a device Cholesky); ``fit="host"`` fits with sklearn exactly
as the reference does and uploads the fitted model once.  Every inference call runs on the GPU either way.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from .gp import DeviceGP


class HeadingTrackingPolicy:
    """The GP-corrected heading controller as an in-kernel policy of ``VecMREnv.rollout`` (``LearningModule.tracking_policy``).

    Per env and step k, from the position p at the start of the step: vd = ref[k, 2:] + gain * (ref[k, :2] - p), then the
    heading search of ``LearningModule.predict_batch`` for vd, action (freq, alpha).  Every operation of vd is rounded on its
    own, so that same torch expression gives the same bits.  gain = 0 is the open-loop correction of main.py (vd = v_ref)."""

    def __init__(self, cheb, a0, freq, Dx, Dy, ref, gain):
        self.cheb = cheb                     # [2, n_coef] verified Chebyshev series of the two GP means on [-pi, pi]
        self.a0, self.freq, self.Dx, self.Dy = float(a0), float(freq), float(Dx), float(Dy)
        self.ref = ref                       # [K, 4] fp64: x_ref, y_ref (start of step k), vx_ref, vy_ref
        self.gain = float(gain)

    @property
    def k_steps(self):
        return self.ref.shape[0]

    def c_policy(self, device):
        """The mr_gp_heading_policy struct for a launch on ``device`` and the tensors it points into (keep them alive)."""
        from . import _lib as L
        cheb, ref = self.cheb.to(device).contiguous(), self.ref.to(device).contiguous()
        pol = L.GpHeadingPolicy(cheb[0].data_ptr(), cheb[1].data_ptr(), cheb.shape[1], 0, self.a0, self.freq, self.Dx,
                                self.Dy, ref.data_ptr(), self.gain)
        return pol, (cheb, ref)


class LearningModule:
    spectral_variance = True     # evaluate GP variances through the low-rank spectral projection when it is exact to 1e-9
    heading_surrogate = True     # search corrected headings on verified Chebyshev interpolants of the two GP means

    def __init__(self, device="cuda", fit="device", preprocess=None):
        """fit: "device" | "host" (sklearn).  preprocess: "device" | "host" (numpy/scipy as in the reference); defaults to
        where the fit runs."""
        self.preprocess = preprocess if preprocess is not None else fit
        if self.preprocess not in ("device", "host"):
            raise ValueError("preprocess must be 'device' or 'host'")
        if fit == "device":
            from .gpr import DeviceGPR
            # Learning_module.py:30-33: RBF(1.0, (1e-2, 10)) + WhiteKernel() (noise 1.0, bounds (1e-5, 1e5)), 5 restarts
            self.gprX = DeviceGPR(n_restarts_optimizer=5, device=device)
            self.gprY = DeviceGPR(n_restarts_optimizer=5, device=device)
        elif fit == "host":
            from sklearn.gaussian_process import GaussianProcessRegressor
            from sklearn.gaussian_process.kernels import RBF, WhiteKernel
            kernel = RBF(length_scale=1.0, length_scale_bounds=(1e-2, 10.0)) + WhiteKernel()     # Learning_module.py:30
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
        self.freq = 0
        self._dx = self._dy = None

    # ---- host-side preprocessing, as in the reference ------------------------------------------
    @staticmethod
    def _velocities(px, py, time):
        from scipy.ndimage import uniform_filter1d
        N = int(1 / 0.035 / 2)                                   # Learning_module.py:47,74
        px = uniform_filter1d(px, N, mode="nearest")
        py = uniform_filter1d(py, N, mode="nearest")
        vx = uniform_filter1d(np.gradient(px, time), int(N / 2), mode="nearest")
        vy = uniform_filter1d(np.gradient(py, time), int(N / 2), mode="nearest")
        return N, px, py, vx, vy

    def _device_preprocess(self, px, py, time, alpha_sim=None, freq=1.0, n_valid=None, subtract_t0=False):
        """mr_learn_preprocess: the filters, gradient, drift means, a0 and GP targets on the device."""
        import ctypes as C

        from . import _lib as L
        lib = L.load()
        dev = torch.device(self.device)
        to = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64) if not torch.is_tensor(a) else a).to(device=dev, dtype=torch.float64).contiguous()
        px, py, time = to(px), to(py), to(time)
        n = int(px.numel())
        N = int(1 / 0.035 / 2)                                   # Learning_module.py:47,74
        vx, vy = torch.empty_like(px), torch.empty_like(px)
        scal = torch.zeros(4, dtype=torch.float64, device=dev)
        ws = torch.empty(4 * n, dtype=torch.float64, device=dev)
        al = to(alpha_sim) if alpha_sim is not None else None
        n_valid = n if n_valid is None else int(n_valid)
        m = max(n_valid - 2 * N, 0)
        X, Yx, Yy = (torch.empty(m, dtype=torch.float64, device=dev) for _ in range(3))
        with torch.cuda.device(dev):
            rc = lib.mr_learn_preprocess(px.data_ptr(), py.data_ptr(), time.data_ptr(), n, N, 1 if subtract_t0 else 0,
                                         float(self.Dx), float(self.Dy), al.data_ptr() if al is not None else None, float(freq),
                                         n_valid, vx.data_ptr(), vy.data_ptr(), X.data_ptr(), Yx.data_ptr(), Yy.data_ptr(),
                                         scal.data_ptr(), ws.data_ptr(), ws.numel() * 8,
                                         C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        L.check(rc, "mr_learn_preprocess")
        return N, vx, vy, X, Yx, Yy, scal

    def estimateDisturbance(self, px, py, time):
        """Learning_module.py:46-59: drift = mean filtered velocity of an idle run."""
        if getattr(self, "preprocess", "host") == "device":
            *_, scal = self._device_preprocess(px, py, time)
            self.Dx, self.Dy = (float(v) for v in scal[:2].cpu())
            return
        N, _, _, vx, vy = self._velocities(np.asarray(px, float), np.asarray(py, float), np.asarray(time, float))
        self.Dx = np.mean(vx[N:-N])
        self.Dy = np.mean(vy[N:-N])

    def learn(self, px, py, alpha_sim, time, actions):
        """Learning_module.py:63-140: a0 estimate + two GPR fits (host), then upload to the device."""
        actions = np.asarray(actions, float)
        freq = actions[0, 0]
        alpha = actions[:, 1]
        if getattr(self, "preprocess", "host") == "device":
            off = np.argwhere(alpha >= 500)                      # controller-off frames, :89-100
            n_valid = int(off[0]) - 1 if len(off) > 0 else None
            _, _, _, X, Yx, Yy, scal = self._device_preprocess(px, py, time, alpha_sim, freq, n_valid, subtract_t0=True)
            a0 = float(scal[2].cpu())
            X = X.reshape(-1, 1)
            self.X, self.Yx, self.Yy = X.cpu().numpy(), Yx.cpu().numpy(), Yy.cpu().numpy()
            if hasattr(self.gprX, "device_model"):               # DeviceGPR takes device tensors as they are
                self.gprX.fit(X, Yx)
                self.gprY.fit(X, Yy)
            else:
                self.gprX.fit(self.X, self.Yx)
                self.gprY.fit(self.X, self.Yy)
            self.a0, self.freq = a0, freq
            self.upload()
            return a0
        time = np.asarray(time, float) - time[0]
        N, px, py, vx, vy = self._velocities(np.asarray(px, float), np.asarray(py, float), time)
        speed = np.sqrt((vx - self.Dx) ** 2 + (vy - self.Dy) ** 2)
        alpha_sim = np.asarray(alpha_sim, float)
        off = np.argwhere(alpha >= 500)                          # controller-off frames, :89-100
        if len(off) > 0:
            cut = int(off[0]) - 1
            alpha_sim, vx, vy, speed = alpha_sim[:cut], vx[:cut], vy[:cut], speed[:cut]
        alpha_sim, vx, vy, speed = alpha_sim[N:-N], vx[N:-N], vy[N:-N], speed[N:-N]
        a0 = np.median(speed / freq)
        X = alpha_sim.reshape(-1, 1)
        Yx = vx - a0 * freq * np.cos(alpha_sim)
        Yy = vy - a0 * freq * np.sin(alpha_sim)
        self.gprX.fit(X, Yx)
        self.gprY.fit(X, Yy)
        self.X, self.Yx, self.Yy = X, Yx, Yy
        self.a0, self.freq = a0, freq
        self.upload()
        return a0

    def upload(self):
        """Fitted models into HBM (sklearn fits are copied; device fits already live there)."""
        as_device = lambda g: g.device_model() if hasattr(g, "device_model") else DeviceGP.from_sklearn(g, self.device)
        self._dx = as_device(self.gprX)
        self._dy = as_device(self.gprY)
        if self.spectral_variance:                      # verified against the triangular form before it is used
            self._dx.enable_spectral_variance()
            self._dy.enable_spectral_variance()
        self._cheb = None
        if self.heading_surrogate and self._dx.dim == 1:
            self._build_heading_surrogate()

    def _build_heading_surrogate(self, n_nodes=2048, n_probe=1024, tol=1e-10):
        """Chebyshev interpolants of the two GP means on the search interval [-pi, pi] of LearningModule.predict
        (Learning_module.py:215).  The means are entire functions of the heading (sums of Gaussians of width l), so
        their Chebyshev coefficients fall off like exp(-(k l / pi)^2 / 2); the series is cut where they reach the
        rounding floor of the sampled means.  Accepted only if it reproduces mr_gp_predict at ``n_probe`` random headings to ``tol`` (relative
        to the largest mean), else the search keeps summing the kernel directly.
        LIBRARY CODE, SET-UP ONLY: the discrete cosine transform below is a 2048^2 torch matmul (cuBLAS), once per
        fitted model; the means it transforms and the search that uses the coefficients are the hand-written kernels."""
        dev = torch.device(self.device)
        j = torch.arange(n_nodes, dtype=torch.float64, device=dev)
        t = torch.cos(math.pi * (j + 0.5) / n_nodes)                       # Chebyshev nodes on [-1, 1]
        mx, my = self.gp_batch(t * math.pi, False)
        k = torch.arange(n_nodes, dtype=torch.float64, device=dev)
        basis = torch.cos(math.pi * torch.outer(k, j + 0.5) / n_nodes)    # T_k(t_j); a 2048^2 matrix, built once per model
        coef = torch.stack([basis @ mx, basis @ my]) * (2.0 / n_nodes)
        coef[:, 0] *= 0.5
        mag = coef.abs().max(dim=0).values
        # the coefficients fall to the rounding floor of the sampled means (~1e-15 of the largest) and stay there: cut the
        # series where they last stand clear of that floor
        floor = float(mag[n_nodes // 2:].max())
        keep = torch.nonzero(mag > max(1e-15 * float(mag.max()), 8.0 * floor)).flatten()
        n_coef = int(keep.max()) + 1 if keep.numel() else 1
        if n_coef > n_nodes // 2:                                          # not resolved: a rougher kernel than the grid
            return
        coef = coef[:, :n_coef].contiguous()
        g = torch.Generator(device=dev).manual_seed(1)
        a = (torch.rand(n_probe, generator=g, device=dev, dtype=torch.float64) * 2 - 1) * math.pi
        ex, ey = self.gp_batch(a, False)
        tt = a / math.pi
        Tk = torch.cos(torch.outer(torch.arange(n_coef, dtype=torch.float64, device=dev), torch.acos(tt.clamp(-1, 1))))
        err = max(float((coef[0] @ Tk - ex).abs().max()), float((coef[1] @ Tk - ey).abs().max()))
        scale = max(float(ex.abs().max()), float(ey.abs().max()), 1e-300)
        if err <= tol * scale:
            self._cheb = coef

    def set_models(self, gprX, gprY, a0, freq, Dx=0.0, Dy=0.0):
        """Install already-fitted GPRs (sklearn or DeviceGPR; e.g. fixed kernels, optimizer=None)."""
        self.gprX, self.gprY, self.a0, self.freq, self.Dx, self.Dy = gprX, gprY, a0, freq, Dx, Dy
        self.X = gprX.X_train_
        self.upload()

    # ---- batched device inference ------------------------------------------------------------------
    def gp_batch(self, alpha, return_std=True):
        """GP posterior at headings alpha [N] -> (muX, muY[, sigX, sigY]) device tensors."""
        if return_std:
            mx, sx = self._dx.predict(alpha, True)
            my, sy = self._dy.predict(alpha, True)
            return mx, my, sx, sy
        return self._dx.predict(alpha), self._dy.predict(alpha)

    def error_batch(self, vd):
        """LearningModule.error for vd [N, 2] (device tensor)."""
        vd = torch.as_tensor(vd, dtype=torch.float64, device=self.device)
        return self.gp_batch(torch.atan2(vd[:, 1], vd[:, 0]), True)

    def velocity_model(self, f, alpha):
        """v_pred = a0*f*[cos a, sin a] + [muX, muY]  (main.py:154-155), batched."""
        alpha = torch.as_tensor(alpha, dtype=torch.float64, device=self.device)
        f = torch.as_tensor(f, dtype=torch.float64, device=self.device)
        mx, my = self.gp_batch(alpha, False)
        return self.a0 * f * torch.cos(alpha) + mx, self.a0 * f * torch.sin(alpha) + my

    # ---- the reference's scalar surface ----------------------------------------------------------------
    def error(self, vd):
        """Learning_module.py:186-196 -> (muX, muY, sigX, sigY), each shape (1,)."""
        a = torch.tensor([math.atan2(vd[1], vd[0])], dtype=torch.float64, device=self.device)
        out = torch.stack(self.gp_batch(a, True)).cpu().numpy()
        return out[0], out[1], out[2], out[3]

    def _objective(self, alpha, vd):
        """objective, Learning_module.py:10-24, with the GP means evaluated on the device."""
        a = torch.tensor([float(alpha)], dtype=torch.float64, device=self.device)
        mu = torch.stack(self.gp_batch(a, False)).cpu().numpy()
        mux, muy = mu[0], mu[1]
        a0f = self.a0 * self.freq
        return (a0f ** 2 + (mux + self.Dx - vd[0]) ** 2 + 2 * a0f * np.cos(alpha) * (mux + self.Dx - vd[0])
                + (muy + self.Dy - vd[1]) ** 2 + 2 * a0f * np.sin(alpha) * (muy + self.Dy - vd[1]))

    def predict_batch(self, vd, return_nfev=False):
        """LearningModule.predict for vd [N, 2] on the device: the bounded minimisation of the objective
        (scipy's algorithm, GP means in the loop) and the posterior at the minimiser.
        Returns (alpha, muX, muY, sigX, sigY) device tensors."""
        import ctypes as C

        from . import _lib as L
        vd = torch.as_tensor(vd, dtype=torch.float64, device=self.device).reshape(-1, 2).contiguous()
        n = vd.shape[0]
        alpha = torch.empty(n, dtype=torch.float64, device=vd.device)
        nfev = torch.empty(n, dtype=torch.int32, device=vd.device)
        stream = C.c_void_p(torch.cuda.current_stream(vd.device).cuda_stream)
        cheb = getattr(self, "_cheb", None)
        if cheb is not None:
            rc = L.load().mr_gp_correct_heading_cheb(cheb[0].data_ptr(), cheb[1].data_ptr(), cheb.shape[1], vd.data_ptr(), n,
                                                     float(self.a0), float(self.freq), float(self.Dx), float(self.Dy),
                                                     alpha.data_ptr(), nfev.data_ptr(), stream)
            L.check(rc, "mr_gp_correct_heading_cheb")
        else:
            rc = L.load().mr_gp_correct_heading(C.byref(self._dx._c), C.byref(self._dy._c), vd.data_ptr(), n, float(self.a0),
                                                float(self.freq), float(self.Dx), float(self.Dy), alpha.data_ptr(),
                                                nfev.data_ptr(), stream)
            L.check(rc, "mr_gp_correct_heading")
        mx, my, sx, sy = self.gp_batch(alpha, True)
        return (alpha, mx, my, sx, sy, nfev) if return_nfev else (alpha, mx, my, sx, sy)

    def tracking_policy(self, ref, gain=0.0):
        """The GP-corrected heading controller for ``VecMREnv.rollout(policy=...)``: ref [K, 4] holds, per control step k,
        the desired position at the start of the step and the desired velocity during it (x_ref, y_ref, vx_ref, vy_ref),
        the same for every env; gain (1/s) feeds the position error back into the desired velocity, 0 = open loop.
        Needs the Chebyshev heading surrogate of this model (built and verified by ``upload``)."""
        if getattr(self, "_cheb", None) is None:
            raise ValueError("tracking_policy needs the verified Chebyshev heading surrogate, which this model does not have; "
                             "compose the controller from predict_batch + VecMREnv.step instead")
        ref = torch.as_tensor(ref).to(device=self.device, dtype=torch.float64).contiguous()
        if ref.dim() != 2 or ref.shape[1] != 4 or ref.shape[0] < 1:
            raise ValueError(f"ref must be [K, 4] (x_ref, y_ref, vx_ref, vy_ref), got {tuple(ref.shape)}")
        if not bool(torch.isfinite(ref).all()):
            raise ValueError("ref must be finite")
        return HeadingTrackingPolicy(self._cheb, self.a0, self.freq, self.Dx, self.Dy, ref, gain)

    def predict(self, vd):
        """Learning_module.py:198-224: bounded scalar minimisation of the objective over alpha, then the
        posterior at the minimiser -> (alpha, muX, muY, sigX, sigY).  Runs entirely on the device."""
        out = torch.stack(self.predict_batch(np.asarray(vd, dtype=np.float64).reshape(1, 2))).cpu().numpy()
        return np.array(out[0, 0]), out[1], out[2], out[3], out[4]
