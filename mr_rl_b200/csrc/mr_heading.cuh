// LearningModule.predict's heading search (Learning_module.py:10-24,198-215), shared by the standalone heading kernels
// (csrc/mr_gp.cu) and the GP-corrected policy of the fused rollout (csrc/mr_rollout.inl).
#pragma once
#include <cuda_runtime.h>

namespace mr {

struct HeadingProblem { double a0f, dx, dy; };

// scipy.optimize._minimize_scalar_bounded (golden section + parabolic interpolation) on [lo, hi]; f is evaluated in the
// order scipy evaluates it.  Returns the minimiser, *nfev = number of objective evaluations.
template <class F>
__device__ __forceinline__ double bounded_minimise(F f, double lo, double hi, double xatol, int maxfun, int* nfev) {
    const double sqrt_eps = sqrt(2.2e-16);
    const double golden_mean = 0.5 * (3.0 - sqrt(5.0));
    double a = lo, b = hi;
    double fulc = a + golden_mean * (b - a);
    double nfc = fulc, xf = fulc;
    double rat = 0.0, e = 0.0;
    double x = xf;
    double fx = f(x);
    int num = 1;
    double ffulc = fx, fnfc = fx;
    double xm = 0.5 * (a + b);
    double tol1 = sqrt_eps * fabs(xf) + xatol / 3.0;
    double tol2 = 2.0 * tol1;
    while (fabs(xf - xm) > (tol2 - 0.5 * (b - a))) {
        bool golden = true;
        if (fabs(e) > tol1) {                                   // try a parabolic fit
            golden = false;
            double r = (xf - nfc) * (fx - ffulc);
            double q = (xf - fulc) * (fx - fnfc);
            double p = (xf - fulc) * q - (xf - nfc) * r;
            q = 2.0 * (q - r);
            if (q > 0.0) p = -p;
            q = fabs(q);
            r = e;
            e = rat;
            if ((fabs(p) < fabs(0.5 * q * r)) && (p > q * (a - xf)) && (p < q * (b - xf))) {
                rat = (p + 0.0) / q;
                x = xf + rat;
                if (((x - a) < tol2) || ((b - x) < tol2)) {
                    const double dm = xm - xf;
                    const double si = (dm > 0.0 ? 1.0 : (dm < 0.0 ? -1.0 : 0.0)) + (dm == 0.0 ? 1.0 : 0.0);
                    rat = tol1 * si;
                }
            } else {
                golden = true;
            }
        }
        if (golden) {                                           // golden-section step
            e = (xf >= xm) ? a - xf : b - xf;
            rat = golden_mean * e;
        }
        const double si = (rat > 0.0 ? 1.0 : (rat < 0.0 ? -1.0 : 0.0)) + (rat == 0.0 ? 1.0 : 0.0);
        x = xf + si * fmax(fabs(rat), tol1);
        const double fu = f(x);
        ++num;
        if (fu <= fx) {
            if (x >= xf) a = xf; else b = xf;
            fulc = nfc; ffulc = fnfc;
            nfc = xf; fnfc = fx;
            xf = x; fx = fu;
        } else {
            if (x < xf) a = x; else b = x;
            if ((fu <= fnfc) || (nfc == xf)) {
                fulc = nfc; ffulc = fnfc;
                nfc = x; fnfc = fu;
            } else if ((fu <= ffulc) || (fulc == xf) || (fulc == nfc)) {
                fulc = x; ffulc = fu;
            }
        }
        xm = 0.5 * (a + b);
        tol1 = sqrt_eps * fabs(xf) + xatol / 3.0;
        tol2 = 2.0 * tol1;
        if (num >= maxfun) break;
    }
    *nfev = num;
    return xf;
}

// The objective at heading alpha with the two GP means given as Chebyshev series on the search interval: s_c holds the
// coefficients as interleaved (x, y) pairs, t = (alpha - mid) * inv_half maps the interval onto [-1, 1].
__device__ __forceinline__ double cheb_heading_objective(double alpha, double vdx, double vdy, const HeadingProblem& hp,
                                                        const double* s_c, int n_coef, double mid, double inv_half) {
    const double t = (alpha - mid) * inv_half, t2 = 2.0 * t;
    double bx1 = 0.0, bx2 = 0.0, by1 = 0.0, by2 = 0.0;       // Clenshaw: b_k = c_k + 2 t b_{k+1} - b_{k+2}
    for (int k = n_coef - 1; k >= 1; --k) {
        const double2 c = *reinterpret_cast<const double2*>(s_c + 2 * k);
        const double nx = fma(t2, bx1, c.x - bx2), ny = fma(t2, by1, c.y - by2);
        bx2 = bx1; bx1 = nx; by2 = by1; by1 = ny;
    }
    const double mux = fma(t, bx1, s_c[0] - bx2), muy = fma(t, by1, s_c[1] - by2);
    const double ex = mux + hp.dx - vdx, ey = muy + hp.dy - vdy;
    double s, c;
    sincos(alpha, &s, &c);
    return hp.a0f * hp.a0f + ex * ex + 2 * hp.a0f * c * ex + ey * ey + 2 * hp.a0f * s * ey;
}

}  // namespace mr
