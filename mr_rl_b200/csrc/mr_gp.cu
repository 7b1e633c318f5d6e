// Gaussian-process inference for Learning_module's disturbance model (sklearn GPR.predict with
// kernel RBF(l) + WhiteKernel(noise), normalize_y=False) and the standalone DDPG actor forward.
//
//   K_q[i][j]  = exp(-0.5 * |q_i/l - X_j/l|^2)                (kernels.RBF.__call__)
//   mean[i]    = sum_j K_q[i][j] * alpha_[j]                  (_gpr.py: K_trans @ alpha_)
//   V          = L^-1 K_q^T  ->  V[i][r] = sum_{c<=r} Linv[r][c] K_q[i][c]
//   std[i]     = sqrt(max(0, (1 + noise) - sum_r V[i][r]^2))  (_gpr.py: diag - einsum(V.T, V))
//
// Kernel 1 (gp_kq_mean): FP64/SFU pipe; one warp per query row, lanes stride the training
//   points so the K_q row is written coalesced; the mean falls out of the same exps.
// Kernel 2 (gp_var): the variance term is a dense triangular contraction
//   [n_q x n] x [n x n]^T, 2 * n_q * n^2 / 2 flops — the only GEMM-shaped work on the hot path.
//   It runs on the FP64 tensor pipe (mma.sync m8n8k4 f64 = DMMA; tcgen05 has no fp64 kind),
//   128x128 CTA tiles, cp.async double-buffered shared-memory staging, fused square-sum epilogue.
#include <cuda_runtime.h>
#include <math_constants.h>

#include "mr_actor.cuh"
#include "mr_actor_tc.cuh"
#include "mr_common.cuh"
#include "mr_dmma.cuh"
#include "mr_step_tma.cuh"   // mbarrier / cp.async.bulk helpers

namespace mr {

// ---- kernel 1: K_q rows + mean ------------------------------------------------------------
template <int DIM, bool WRITE_KQ>
__global__ void __launch_bounds__(256)
gp_kq_mean_kernel(const double* __restrict__ q, int64_t n_q, const double* __restrict__ xtr /* X_train / l */,
                  const double* __restrict__ alpha, int n_pad, int n_train, double ls,
                  double* __restrict__ kq /*[n_q][n_pad]*/, double* __restrict__ mean) {
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // one warp per query
    if (row >= n_q) return;
    double q0 = q[row * DIM] / ls, q1 = 0.0;             // sklearn: cdist(X / l, Y / l, "sqeuclidean")
    if (DIM == 2) q1 = q[row * DIM + 1] / ls;
    double acc = 0.0;
    double* out = kq + row * (int64_t)n_pad;
    for (int j = lane; j < n_pad; j += 32) {
        double d2;
        if (DIM == 1) { const double d = q0 - xtr[j]; d2 = d * d; }
        else { const double d0 = q0 - xtr[2 * j], d1 = q1 - xtr[2 * j + 1]; d2 = d0 * d0 + d1 * d1; }
        double k = exp(-0.5 * d2);
        if (j >= n_train) k = 0.0;                       // padding contributes nothing
        if (WRITE_KQ) out[j] = k;
        acc = fma(k, alpha[j], acc);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) mean[row] = acc;
}



// exp(x) for x <= 0 with a 64-entry table of 2^(j/64) in shared memory and a degree-5 polynomial:
// x = (64 m + j) ln2/64 + r, |r| <= ln2/128, exp(x) = 2^m * T[j] * (1 + r + ... + r^5/120) (truncation
// 3.5e-17).  ~14 fp64 instructions instead of the ~25 of the library exp; ~2 ulp.  Results below
// 2^-1021 flush to 0 (such kernel values cannot influence a sum whose other terms are O(1e-300) larger).
__device__ __forceinline__ void exp_table_init(double* T) {
    if (threadIdx.x < 64) T[threadIdx.x] = exp2((double)threadIdx.x / 64.0);
}
__device__ __forceinline__ double exp_neg_tab(double x, const double* __restrict__ T) {
    const double t = x * 92.33248261689366;                      // 64 / ln 2
    const int n = __double2int_rn(t);
    const double nd = (double)n;
    double r = fma(-nd, 0x1.62e42fefa0000p-7, x);                // ln2/64, high 36 bits (n * hi is exact)
    r = fma(-nd, 0x1.cf78000000000p-46, r);                      // ... and the remainder
    double p = fma(r, 1.0 / 120.0, 1.0 / 24.0);
    p = fma(p, r, 1.0 / 6.0);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    const int m = n >> 6;                                        // floor division: j = n & 63 in [0, 63]
    const double v = T[n & 63] * p;                              // in [1, 2.04)
    if (m < -1021) return 0.0;
    return __longlong_as_double(__double_as_longlong(v) + ((long long)m << 52));
}

// ---- kernel 1 (staged): training points and alpha live in shared memory ---------------------
// Persistent CTAs: the (pre-scaled) training inputs and alpha_ are fetched ONCE per CTA with two TMA
// bulk copies (cp.async.bulk + mbarrier), then every warp walks over query rows, QPW rows at a time,
// lanes striding the training points (conflict-free LDS.64), and reduces with xor shuffles.
template <int DIM, bool WRITE_KQ, int QPW>
__global__ void __launch_bounds__(256)
gp_kq_mean_smem_kernel(const double* __restrict__ q, int64_t n_q, const double* __restrict__ xtr,
                       const double* __restrict__ alpha, int n_pad, double ls, double* __restrict__ kq,
                       double* __restrict__ mean) {
    extern __shared__ __align__(128) unsigned char gp_smem[];
    double* s_x = reinterpret_cast<double*>(gp_smem);                 // [n_pad][DIM]
    double* s_a = s_x + (size_t)n_pad * DIM;                          // [n_pad]
    double* s_tab = s_a + n_pad;                                      // [64] 2^(j/64)
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_tab + 64);
    exp_table_init(s_tab);
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t bx = (uint32_t)n_pad * DIM * 8u, ba = (uint32_t)n_pad * 8u;
        mbar_expect_tx(bar, bx + ba);
        bulk_load(s_x, xtr, bx, bar);
        bulk_load(s_a, alpha, ba, bar);
    }
    mbar_wait(bar, 0);

    const int lane = threadIdx.x & 31;
    const int warps_total = (int)(gridDim.x * (blockDim.x >> 5));
    const int warp_global = (int)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));
    for (int64_t row0 = (int64_t)warp_global * QPW; row0 < n_q; row0 += (int64_t)warps_total * QPW) {
        double q0[QPW], q1[QPW], acc[QPW];
#pragma unroll
        for (int r = 0; r < QPW; ++r) {
            const int64_t row = row0 + r < n_q ? row0 + r : n_q - 1;  // clamp: tail rows recompute the last row
            q0[r] = q[row * DIM] / ls;                                // sklearn: cdist(X / l, Y / l, "sqeuclidean")
            q1[r] = DIM == 2 ? q[row * DIM + 1] / ls : 0.0;
            acc[r] = 0.0;
        }
        for (int j = lane; j < n_pad; j += 32) {
            const double a = s_a[j];
            double x0, x1 = 0.0;
            if (DIM == 1) x0 = s_x[j]; else { x0 = s_x[2 * j]; x1 = s_x[2 * j + 1]; }
#pragma unroll
            for (int r = 0; r < QPW; ++r) {
                const double d0 = q0[r] - x0;
                double d2 = d0 * d0;
                if (DIM == 2) { const double d1 = q1[r] - x1; d2 = fma(d1, d1, d2); }
                const double k = exp_neg_tab(-0.5 * d2, s_tab);       // padding columns meet alpha = 0 / zero linv columns
                if (WRITE_KQ && row0 + r < n_q) kq[(row0 + r) * (int64_t)n_pad + j] = k;
                acc[r] = fma(k, a, acc[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < QPW; ++r) {
            double v = acc[r];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            if (lane == 0 && row0 + r < n_q) mean[row0 + r] = v;
        }
    }
}

// launch helper: staged kernel when the model fits in shared memory, else the global-memory kernel
template <int DIM, bool WRITE_KQ>
static void launch_kq_mean(const double* q, int64_t n_q, const mr_gp_model* gp, double* kq, double* mean, cudaStream_t s) {
    const size_t smem = (size_t)gp->n_pad * (DIM + 1) * 8 + 64 * 8 + 16;
    const bool aligned = (((uintptr_t)gp->x_train_scaled | (uintptr_t)gp->alpha) & 15u) == 0;   // TMA bulk copies
    if (smem <= 200 * 1024 && aligned) {
        constexpr int QPW = 4;
        static int sms[kMaxDevices] = {};
        const int dev = current_device();
        if (!sms[dev]) { cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev); if (sms[dev] <= 0) sms[dev] = 148; }
        cudaFuncSetAttribute(gp_kq_mean_smem_kernel<DIM, WRITE_KQ, QPW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        int per_sm = (int)((220 * 1024) / (smem + 1024));
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 4) per_sm = 4;
        int64_t want = (n_q + 8 * QPW - 1) / (8 * QPW);             // CTAs needed if every warp took one pass
        int64_t grid = (int64_t)sms[dev] * per_sm;
        if (grid > want) grid = want;
        if (grid < 1) grid = 1;
        gp_kq_mean_smem_kernel<DIM, WRITE_KQ, QPW><<<(unsigned)grid, 256, smem, s>>>(q, n_q, gp->x_train_scaled, gp->alpha,
                                                                                     gp->n_pad, gp->length_scale, kq, mean);
    } else {
        const unsigned blocks = (unsigned)((n_q * 32 + 255) / 256);
        gp_kq_mean_kernel<DIM, WRITE_KQ><<<blocks, 256, 0, s>>>(q, n_q, gp->x_train_scaled, gp->alpha, gp->n_pad, gp->n_train,
                                                                gp->length_scale, kq, mean);
    }
}

// ---- kernel 2: triangular contraction + square-sum (mainloop: mr_dmma.cuh) --------------------
__global__ void __launch_bounds__(256)
gp_var_kernel(const double* __restrict__ kq, const double* __restrict__ linv, int n_pad, int64_t n_q_pad,
              double* __restrict__ ssq, int dense) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int warp_m = warp >> 2;
    const int g = lane >> 2, t4 = lane & 3;
    const int bn = (int)gridDim.y - 1 - (int)blockIdx.y;        // heaviest column blocks first
    const int64_t m0 = (int64_t)blockIdx.x * GP_BM;
    const int r0 = bn * GP_BN;
    // triangular L^-1: c <= r, columns beyond the diagonal block are zero; dense spectral projection: all columns
    const int k_tiles = dense ? n_pad / GP_BK : (r0 + GP_BN) / GP_BK;

    double acc[8][4][2];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    dmma_tile_tn(kq + m0 * n_pad, n_pad, linv + (int64_t)r0 * n_pad, n_pad, k_tiles, acc, smem);   // A[m][c], B[r][c]

    // epilogue: sum of squares over this CTA's 128 columns, per query row
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) s += acc[i][j][0] * acc[i][j][0] + acc[i][j][1] * acc[i][j][1];
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        const int64_t row = m0 + warp_m * 64 + i * 8 + g;
        if (t4 == 0 && row < n_q_pad) atomicAdd(ssq + row, s);
    }
}

// ---- fused posterior for the spectral form: mean AND std of 128 queries per CTA in one pass, K_q never leaves the SM ----
// Per 16-column slice of the training set every thread evaluates 8 kernel values (one query row, 8 training points)
// straight into the A tile of the DMMA pipeline (and into its running mean), the B tile (projection rows) streams in
// with cp.async; C = K_q P^T accumulates on the FP64 tensor pipe; the epilogue squares and sums the 128 columns.
// (Training inputs / alpha are read with __ldg: staging them in shared memory per CTA was measured slower at config-3
// size, 5.98 vs 5.59 ms per GP — 2048 CTAs each copying 48 KB costs more than the L1-resident reads.)
// NT = n8 column tiles per warp: the CTA covers 32 NT projection rows per pass (96 rows when ~80 eigenvalues matter)
template <int DIM, int NT>
__global__ void __launch_bounds__(256)
gp_posterior_spectral_kernel(const double* __restrict__ q, int64_t n_q, const double* __restrict__ xs, const double* __restrict__ alpha,
                             const double* __restrict__ proj, int n_pad, int proj_rows, double ls, double diag,
                             double* __restrict__ mean, double* __restrict__ std) {
    extern __shared__ __align__(16) double smem[];
    __shared__ double s_tab[64];
    __shared__ double s_ssq[GP_BM];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int warp_m = warp >> 2, warp_n = warp & 3, g = lane >> 2, t4 = lane & 3;
    exp_table_init(s_tab);
    if (tid < GP_BM) s_ssq[tid] = 0.0;
    const int64_t m0 = (int64_t)blockIdx.x * GP_BM;
    const int my_row = tid >> 1, my_half = tid & 1;            // this thread's query row and 8-column half of a slice
    double qv[DIM];
#pragma unroll
    for (int c = 0; c < DIM; ++c) qv[c] = (m0 + my_row < n_q) ? q[(m0 + my_row) * DIM + c] / ls : 0.0;   // RBF scales both operands
    const int k_tiles = n_pad / GP_BK;
    double mean_acc = 0.0;
    __syncthreads();

    constexpr int BN = 32 * NT;
    for (int rb = 0; rb < proj_rows / BN; ++rb) {
        double acc[8][NT][2];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < NT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        const double* b_src = proj + (int64_t)rb * BN * n_pad;
        auto load_b = [&](int stage, int kt) {                  // BN rows x 16 doubles = 8 BN 16-byte chunks, 256 threads x NT
            double* Bs = smem + stage * GP_STAGE + GP_BM * GP_LD;
#pragma unroll
            for (int it = 0; it < NT; ++it) {
                const int chunk = tid + it * 256;
                const int r = chunk >> 3, cc = (chunk & 7) * 2;
                cp_async16(Bs + r * GP_LD + cc, b_src + (int64_t)r * n_pad + kt * GP_BK + cc);
            }
        };
        auto make_a = [&](int stage, int kt, bool with_mean) {  // kernel values of (my_row, 8 training points)
            double* As = smem + stage * GP_STAGE + my_row * GP_LD + my_half * 8;
            const int c0 = kt * GP_BK + my_half * 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                double d2 = 0.0;
#pragma unroll
                for (int c = 0; c < DIM; ++c) { const double d = qv[c] - __ldg(xs + (int64_t)(c0 + j) * DIM + c); d2 = fma(d, d, d2); }
                const double k = exp_neg_tab(-0.5 * d2, s_tab);
                As[j] = k;
                if (with_mean) mean_acc = fma(k, __ldg(alpha + c0 + j), mean_acc);
            }
        };
        make_a(0, 0, rb == 0);
        load_b(0, 0);
        cp_async_commit();
        if (k_tiles > 1) load_b(1, 1);
        cp_async_commit();
        for (int kt = 0; kt < k_tiles; ++kt) {
            cp_async_wait<GP_STAGES - 2>();
            __syncthreads();                                    // A(kt) written by everyone, B(kt) landed
            if (kt + 2 < k_tiles) load_b((kt + 2) % GP_STAGES, kt + 2);
            cp_async_commit();
            if (kt + 1 < k_tiles) make_a((kt + 1) % GP_STAGES, kt + 1, rb == 0);
            const double* As = smem + (kt % GP_STAGES) * GP_STAGE + (warp_m * 64) * GP_LD;
            const double* Bs = smem + (kt % GP_STAGES) * GP_STAGE + GP_BM * GP_LD + (warp_n * 8 * NT) * GP_LD;
#pragma unroll
            for (int k4 = 0; k4 < GP_BK / 4; ++k4) {
                double a[8], b[NT];
#pragma unroll
                for (int i = 0; i < 8; ++i) a[i] = As[(i * 8 + g) * GP_LD + k4 * 4 + t4];
#pragma unroll
                for (int j = 0; j < NT; ++j) b[j] = Bs[(j * 8 + g) * GP_LD + k4 * 4 + t4];
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < NT; ++j) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
        }
        cp_async_wait<0>();
        __syncthreads();                                        // the ring is reused by the next row block
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < NT; ++j) s += acc[i][j][0] * acc[i][j][0] + acc[i][j][1] * acc[i][j][1];
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            if (t4 == 0) atomicAdd(&s_ssq[warp_m * 64 + i * 8 + g], s);
        }
    }
    mean_acc += __shfl_xor_sync(0xffffffffu, mean_acc, 1);      // the two column halves of a row sit in adjacent lanes
    __syncthreads();
    if (my_half == 0 && m0 + my_row < n_q) {
        mean[m0 + my_row] = mean_acc;
        double v = diag - s_ssq[my_row];
        if (v < 0.0) v = 0.0;                                   // sklearn clips negative variances to 0
        std[m0 + my_row] = sqrt(v);
    }
}

__global__ void gp_std_finish_kernel(const double* __restrict__ ssq, int64_t n_q, double diag, double* __restrict__ std) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_q) return;
    double v = diag - ssq[i];
    if (v < 0.0) v = 0.0;                                      // sklearn clips negative variances to 0
    std[i] = sqrt(v);
}


// ---- LearningModule.predict: batched bounded scalar minimisation with the GP means in the loop ----
// One warp per desired velocity.  The control flow is scipy's _minimize_scalar_bounded (golden section
// + parabolic interpolation, xatol = 1e-5, maxiter = 500) on bounds [-pi, pi], evaluated redundantly
// by all lanes; each objective call (Learning_module.py:10-24) needs the two GP posterior means, which
// the 32 lanes compute cooperatively (lane-strided training points, xor-shuffle reduction).
struct HeadingProblem { double a0f, dx, dy; };

__device__ __forceinline__ double gp_objective_warp(double alpha, double vdx, double vdy, const HeadingProblem& hp,
                                                    const double* __restrict__ xsx, const double* __restrict__ ax,
                                                    double lsx, const double* __restrict__ xsy,
                                                    const double* __restrict__ ay, double lsy, int n_pad, int n_train,
                                                    int lane, const double* __restrict__ tab) {
    const double qx = alpha / lsx, qy = alpha / lsy;
    double sx = 0.0, sy = 0.0;
    for (int j = lane; j < n_pad; j += 32) {
        const double d0 = qx - xsx[j], d1 = qy - xsy[j];
        double kx = exp_neg_tab(-0.5 * (d0 * d0), tab), ky = exp_neg_tab(-0.5 * (d1 * d1), tab);
        if (j >= n_train) { kx = 0.0; ky = 0.0; }
        sx = fma(kx, ax[j], sx);
        sy = fma(ky, ay[j], sy);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        sx += __shfl_xor_sync(0xffffffffu, sx, off);
        sy += __shfl_xor_sync(0xffffffffu, sy, off);
    }
    const double ex = sx + hp.dx - vdx, ey = sy + hp.dy - vdy;     // mux + Dx - v_d[0], muy + Dy - v_d[1]
    double s, c;
    sincos(alpha, &s, &c);
    return hp.a0f * hp.a0f + ex * ex + 2 * hp.a0f * c * ex + ey * ey + 2 * hp.a0f * s * ey;
}

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

__global__ void __launch_bounds__(256)
gp_correct_heading_kernel(const double* __restrict__ vd, int64_t n, HeadingProblem hp, const double* __restrict__ xsx,
                          const double* __restrict__ ax, double lsx, const double* __restrict__ xsy,
                          const double* __restrict__ ay, double lsy, int n_pad, int n_train, double lo, double hi,
                          double xatol, int maxfun, double* __restrict__ alpha_out, int32_t* __restrict__ nfev_out) {
    __shared__ double s_tab[64];
    exp_table_init(s_tab);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n) return;
    const double vdx = vd[2 * row], vdy = vd[2 * row + 1];
    auto f = [&](double x) { return gp_objective_warp(x, vdx, vdy, hp, xsx, ax, lsx, xsy, ay, lsy, n_pad, n_train, lane, s_tab); };
    int num = 0;
    const double xf = bounded_minimise(f, lo, hi, xatol, maxfun, &num);
    if (lane == 0) {
        alpha_out[row] = xf;
        if (nfev_out) nfev_out[row] = num;
    }
}

// The same search with the two GP means replaced by their Chebyshev interpolants on [lo, hi] (the search interval): a GP
// mean with an RBF kernel is an entire function of the heading, ~150 coefficients reproduce it to the accuracy of the
// direct sum, and one Clenshaw pass costs ~300 FMAs instead of 2 x 2000 exponentials.  One thread per velocity.  The
// caller builds and VERIFIES the interpolants against mr_gp_predict before using this kernel.
__global__ void __launch_bounds__(128)
gp_correct_heading_cheb_kernel(const double* __restrict__ vd, int64_t n, HeadingProblem hp, const double* __restrict__ cx,
                               const double* __restrict__ cy, int n_coef, double lo, double hi, double xatol, int maxfun,
                               double* __restrict__ alpha_out, int32_t* __restrict__ nfev_out) {
    extern __shared__ __align__(16) double s_c[];                // [2][n_coef] interleaved (x, y)
    for (int k = threadIdx.x; k < n_coef; k += blockDim.x) { s_c[2 * k] = cx[k]; s_c[2 * k + 1] = cy[k]; }
    __syncthreads();
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    const double vdx = vd[2 * row], vdy = vd[2 * row + 1];
    const double mid = 0.5 * (lo + hi), inv_half = 2.0 / (hi - lo);
    auto f = [&](double alpha) {
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
    };
    int num = 0;
    const double xf = bounded_minimise(f, lo, hi, xatol, maxfun, &num);
    alpha_out[row] = xf;
    if (nfev_out) nfev_out[row] = num;
}

// ---- LearningModule2D.predict: batched box-constrained least squares over (alpha, f) --------
// Learning_module_2d.py:11-25 minimises (a0 f)^2 + (muX - vd0)^2 + 2 a0 f cos(alpha) (muX - vd0) + (muY - vd1)^2 + ...,
// which is exactly |r|^2 for r(alpha, f) = a0 f (cos alpha, sin alpha) + (muX, muY)(alpha, f) - vd.  One warp per desired
// velocity; one PASS evaluates, at a trial point, both GP means with their gradients and Hessians (lanes stride the
// training points, xor-shuffle reduction: 6 sums per GP), so r, its Jacobian J and the Hessian of |r|^2 / 2,
// H = J^T J + r0 d2(r0) + r1 d2(r1), come out of one pass.  The solver is a projected Newton method with
// Levenberg-Marquardt damping (Nielsen's update), held redundantly by all lanes:
//   - a coordinate on a bound whose gradient g = J^T r points out of the box is held fixed; the damped 2x2 (or 1x1)
//     system is solved on the free coordinates and the trial point is clipped to the box;
//   - a trial is accepted if |r|^2 decreases; each trial is one pass;
//   - converged (status 0) when the projected gradient |x - clip(x - g)|_inf <= kAction2dGtol (1 + |vd|^2), or the
//     next step is at rounding level; kAction2dMaxPass passes -> status 1 with the best point so far;
//   - a non-finite vd, or non-finite means at the start point -> x = NaN, status 2.
// The curvature terms r.d2r matter where the minimum is not a root (f on a bound, low speeds): with J^T J alone the
// solver converges only linearly there (30-60 passes against 7-20 with them in a numpy model of this solver).
// The exponentials use the table form the staged mr_gp_predict kernel uses, in the same order per lane.
constexpr double kAction2dGtol = 1e-12;
constexpr int kAction2dMaxPass = 64;

struct GpMoments2 { double m, s0, s1, s00, s01, s11; };   // sum a_j k_j (1, s, s s^T) with s_j = q / l - X_j / l

__device__ __forceinline__ void gp_moments_2d_warp(double q0, double q1, const double* __restrict__ xsx,
                                                   const double* __restrict__ ax, double lsx, const double* __restrict__ xsy,
                                                   const double* __restrict__ ay, double lsy, int n_train, int lane,
                                                   const double* __restrict__ tab, GpMoments2& mx, GpMoments2& my) {
    const double px0 = q0 / lsx, px1 = q1 / lsx, py0 = q0 / lsy, py1 = q1 / lsy;
    double v[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) v[i] = 0.0;
    for (int j = lane; j < n_train; j += 32) {
        const double dx0 = px0 - xsx[2 * j], dx1 = px1 - xsx[2 * j + 1];
        const double dy0 = py0 - xsy[2 * j], dy1 = py1 - xsy[2 * j + 1];
        double d2x = dx0 * dx0, d2y = dy0 * dy0;
        d2x = fma(dx1, dx1, d2x);
        d2y = fma(dy1, dy1, d2y);
        const double kx = exp_neg_tab(-0.5 * d2x, tab), ky = exp_neg_tab(-0.5 * d2y, tab);
        const double ajx = ax[j], ajy = ay[j];
        v[0] = fma(kx, ajx, v[0]);
        v[6] = fma(ky, ajy, v[6]);
        const double wx = kx * ajx, wy = ky * ajy;
        const double wx0 = wx * dx0, wy0 = wy * dy0, wx1 = wx * dx1, wy1 = wy * dy1;
        v[1] += wx0; v[2] += wx1; v[3] = fma(wx0, dx0, v[3]); v[4] = fma(wx0, dx1, v[4]); v[5] = fma(wx1, dx1, v[5]);
        v[7] += wy0; v[8] += wy1; v[9] = fma(wy0, dy0, v[9]); v[10] = fma(wy0, dy1, v[10]); v[11] = fma(wy1, dy1, v[11]);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
#pragma unroll
        for (int i = 0; i < 12; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], off);
    mx = GpMoments2{v[0], v[1], v[2], v[3], v[4], v[5]};
    my = GpMoments2{v[6], v[7], v[8], v[9], v[10], v[11]};
}

struct Action2dState { double r0, r1, g0, g1, h00, h01, h11, F; };

// residual, gradient g = J^T r and Hessian H of |r|^2 / 2 at (alpha, f) from the two GPs' moments
__device__ __forceinline__ Action2dState action_2d_state(double alpha, double f, double vd0, double vd1, double a0,
                                                         const GpMoments2& mx, double lsx, const GpMoments2& my, double lsy) {
    double sa, ca;
    sincos(alpha, &sa, &ca);
    const double a0f = a0 * f;
    Action2dState st;
    st.r0 = fma(a0f, ca, mx.m) - vd0;
    st.r1 = fma(a0f, sa, my.m) - vd1;
    // d mu / d q = -S / l ;  d2 mu / dq dq^T = (S2 - mu I) / l^2
    const double ix = 1.0 / lsx, iy = 1.0 / lsy;
    const double j00 = -a0f * sa - mx.s0 * ix, j01 = a0 * ca - mx.s1 * ix;
    const double j10 = a0f * ca - my.s0 * iy, j11 = a0 * sa - my.s1 * iy;
    st.g0 = j00 * st.r0 + j10 * st.r1;
    st.g1 = j01 * st.r0 + j11 * st.r1;
    const double cx = st.r0 * ix * ix, cy = st.r1 * iy * iy;
    const double c00 = cx * (mx.s00 - mx.m) + cy * (my.s00 - my.m) - a0f * (st.r0 * ca + st.r1 * sa);
    const double c01 = cx * mx.s01 + cy * my.s01 + a0 * (st.r1 * ca - st.r0 * sa);
    const double c11 = cx * (mx.s11 - mx.m) + cy * (my.s11 - my.m);
    st.h00 = j00 * j00 + j10 * j10 + c00;
    st.h01 = j00 * j01 + j10 * j11 + c01;
    st.h11 = j01 * j01 + j11 * j11 + c11;
    st.F = st.r0 * st.r0 + st.r1 * st.r1;
    return st;
}

__global__ void __launch_bounds__(256)
gp_correct_action_2d_kernel(const double* __restrict__ vd, int64_t n, double a0, const double* __restrict__ xsx,
                            const double* __restrict__ ax, double lsx, const double* __restrict__ xsy,
                            const double* __restrict__ ay, double lsy, int n_train, double lo0, double lo1, double hi0,
                            double hi1, double* __restrict__ x_out, int32_t* __restrict__ iters_out,
                            uint8_t* __restrict__ status_out) {
    __shared__ double s_tab[64];
    exp_table_init(s_tab);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n) return;
    const double vd0 = vd[2 * row], vd1 = vd[2 * row + 1];
    auto clip0 = [&](double v) { return fmin(fmax(v, lo0), hi0); };
    auto clip1 = [&](double v) { return fmin(fmax(v, lo1), hi1); };
    auto eval = [&](double alpha, double f) {
        GpMoments2 mx, my;
        gp_moments_2d_warp(alpha, f, xsx, ax, lsx, xsy, ay, lsy, n_train, lane, s_tab, mx, my);
        return action_2d_state(alpha, f, vd0, vd1, a0, mx, lsx, my, lsy);
    };
    double x0 = CUDART_NAN, x1 = CUDART_NAN;
    int passes = 0, status = 2;
    if (isfinite(vd0) && isfinite(vd1)) {
        // Learning_module_2d.py:229-230 (_desired), clipped into the box as L-BFGS-B clips its x0
        x0 = clip0(atan2(vd1, vd0));
        x1 = clip1(sqrt(fma(vd1, vd1, vd0 * vd0)) / a0);
        Action2dState s = eval(x0, x1);
        passes = 1;
        if (!isfinite(s.F)) {
            x0 = x1 = CUDART_NAN;
        } else {
            const double gtol = kAction2dGtol * (1.0 + fma(vd1, vd1, vd0 * vd0));
            const double step_eps = 0x1p-50;
            double mu = 1e-3 * fmax(fmax(fabs(s.h00), fabs(s.h11)), 1e-300), nu = 2.0;
            status = -1;
            while (status < 0) {
                const double pg = fmax(fabs(x0 - clip0(x0 - s.g0)), fabs(x1 - clip1(x1 - s.g1)));
                if (pg <= gtol) { status = 0; break; }
                const bool free0 = !((x0 <= lo0 && s.g0 > 0.0) || (x0 >= hi0 && s.g0 < 0.0));
                const bool free1 = !((x1 <= lo1 && s.g1 > 0.0) || (x1 >= hi1 && s.g1 < 0.0));
                for (;;) {                                         // damped trials until one is accepted
                    if (!(mu <= 1e300)) { status = 1; break; }    // only a non-finite Hessian gets here
                    double d0 = 0.0, d1 = 0.0;
                    const double a00 = s.h00 + mu, a11 = s.h11 + mu;
                    if (free0 && free1) {
                        const double det = a00 * a11 - s.h01 * s.h01;
                        if (!(det > 0.0 && a00 > 0.0)) { mu *= nu; nu *= 2.0; continue; }   // not positive definite yet
                        d0 = (s.h01 * s.g1 - a11 * s.g0) / det;
                        d1 = (s.h01 * s.g0 - a00 * s.g1) / det;
                    } else if (free0) {
                        if (!(a00 > 0.0)) { mu *= nu; nu *= 2.0; continue; }
                        d0 = -s.g0 / a00;
                    } else {                                       // pg > 0 leaves at least one coordinate free
                        if (!(a11 > 0.0)) { mu *= nu; nu *= 2.0; continue; }
                        d1 = -s.g1 / a11;
                    }
                    const double t0 = clip0(x0 + d0), t1 = clip1(x1 + d1);
                    const double h0 = t0 - x0, h1 = t1 - x1;
                    if (fabs(h0) <= step_eps * (1.0 + fabs(x0)) && fabs(h1) <= step_eps * (1.0 + fabs(x1))) { status = 0; break; }
                    if (passes >= kAction2dMaxPass) { status = 1; break; }
                    const Action2dState t = eval(t0, t1);
                    ++passes;
                    if (t.F < s.F) {
                        // gain ratio against the quadratic model of |r|^2 / 2 along the (clipped) step
                        const double pred = -(s.g0 * h0 + s.g1 * h1) - 0.5 * (h0 * h0 * s.h00 + 2.0 * h0 * h1 * s.h01 + h1 * h1 * s.h11);
                        const double rho = pred > 0.0 ? 0.5 * (s.F - t.F) / pred : 0.0;
                        const double c = 2.0 * rho - 1.0;
                        mu *= fmax(1.0 / 3.0, 1.0 - c * c * c);
                        nu = 2.0;
                        x0 = t0; x1 = t1; s = t;
                        break;
                    }
                    mu *= nu; nu *= 2.0;                            // rejected (also when t.F is NaN)
                }
            }
        }
    }
    if (lane == 0) {
        x_out[2 * row] = x0;
        x_out[2 * row + 1] = x1;
        if (iters_out) iters_out[row] = passes;
        if (status_out) status_out[row] = (uint8_t)status;
    }
}

static bool fused_spectral_disabled() {          // MR_GP_FUSED=0: keep the two-kernel path for the spectral form (A/B measurements)
    static const bool off = [] { const char* e = getenv("MR_GP_FUSED"); return e && e[0] == '0'; }();
    return off;
}

constexpr int64_t kGpChunk = 16384;   // queries per pass of the variance pipeline (K_q chunk = chunk * n_pad * 8 B)

static int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

// ---- standalone actor forward -------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(128)
actor_forward_kernel(const float* __restrict__ actor, const T* __restrict__ obs, int64_t stride, int64_t n, float hi0,
                     float hi1, T* __restrict__ actions) {
    extern __shared__ __align__(16) float s_actor[];
    for (int k = threadIdx.x; k < kActorParams; k += blockDim.x) s_actor[k] = actor[k];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float o5[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) o5[k] = (float)obs[k * stride + i];
    float a2[2];
    actor_forward_smem(s_actor, o5, hi0, hi1, a2);
    actions[2 * i] = (T)a2[0];
    actions[2 * i + 1] = (T)a2[1];
}

// The same network for MR_Env observations (goal components obs[2], obs[3] identically zero, MR_env.py:57) with the
// hidden 64 x 64 layer on the tensor cores: persistent CTAs of 128 envs, tcgen05.mma 3xTF32 into TMEM
// (mr_actor_tc.cuh, shared with the fused rollout).  Measured at 2^20 envs: see tools/ddpgbench.py.
template <class T>
__global__ void __launch_bounds__(kTcRows, 1)
actor_forward_tc_kernel(const float* __restrict__ actor, const T* __restrict__ obs, int64_t stride, int64_t n, float hi0,
                        float hi1, T* __restrict__ actions) {
    extern __shared__ __align__(128) unsigned char s_dyn[];
    ActorTcSmem& sm = *reinterpret_cast<ActorTcSmem*>(s_dyn);
    actor_tc_setup(sm, actor);
    __syncthreads();
    const int64_t n_tiles = (n + kTcRows - 1) / kTcRows;
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {     // every thread runs every iteration
        const int64_t i = tile * kTcRows + threadIdx.x;
        const bool live = i < n;
        float o5[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        if (live) { o5[0] = (float)obs[i]; o5[1] = (float)obs[stride + i]; o5[4] = (float)obs[4 * stride + i]; }
        float a2[2];
        actor_tc_forward(sm, o5, hi0, hi1, it, a2);
        if (live) { actions[2 * i] = (T)a2[0]; actions[2 * i + 1] = (T)a2[1]; }
    }
    actor_tc_teardown(sm);
}

}  // namespace mr

extern "C" {

int64_t mr_gp_workspace_bytes(const mr_gp_model* gp, int64_t n_q, int32_t want_std) {
    if (!gp || !want_std || n_q <= 0) return 0;
    const int64_t chunk = mr::round_up(n_q < mr::kGpChunk ? n_q : mr::kGpChunk, mr::GP_BM);
    return chunk * (int64_t)gp->n_pad * 8 + chunk * 8;
}

int mr_gp_predict(const mr_gp_model* gp, const double* q, int64_t n_q, double* mean, double* std, void* workspace,
                  int64_t workspace_bytes, void* stream) {
    mr::NvtxRange nvtx_range("mr_gp_predict");
    using namespace mr;
    if (!gp || !gp->x_train_scaled || !gp->alpha) return fail(MR_ERR_ARG, "mr_gp_predict: null model");
    if (n_q < 0) return fail(MR_ERR_ARG, "mr_gp_predict: bad n_q");
    if (n_q == 0) return MR_OK;
    if (!q || !mean) return fail(MR_ERR_ARG, "mr_gp_predict: null q/mean");
    if (gp->dim != 1 && gp->dim != 2) return fail(MR_ERR_UNSUPPORTED, "mr_gp_predict: dim must be 1 or 2");
    if (gp->n_pad % MR_GP_PAD != 0 || gp->n_train > gp->n_pad || gp->n_train <= 0)
        return fail(MR_ERR_ARG, "mr_gp_predict: n_pad must be a multiple of %d and >= n_train", MR_GP_PAD);
    if (!(gp->length_scale > 0)) return fail(MR_ERR_ARG, "mr_gp_predict: bad length_scale");
    cudaStream_t s = (cudaStream_t)stream;
    if (!std) {
        if (gp->dim == 1) launch_kq_mean<1, false>(q, n_q, gp, nullptr, mean, s);
        else launch_kq_mean<2, false>(q, n_q, gp, nullptr, mean, s);
        return check_launch("mr_gp_predict(mean)");
    }
    if (!gp->linv) return fail(MR_ERR_ARG, "mr_gp_predict: std requested but model has no linv");
    if (gp->proj_rows < 0 || gp->proj_rows % 32 != 0 || gp->proj_rows > gp->n_pad ||
        (gp->proj_rows > MR_GP_PAD && gp->proj_rows % MR_GP_PAD != 0))
        return fail(MR_ERR_ARG, "mr_gp_predict: proj_rows must be 0, 32/64/96/128 or a multiple of %d up to n_pad", MR_GP_PAD);
    if (gp->proj_rows % MR_GP_PAD != 0 && fused_spectral_disabled())
        return fail(MR_ERR_UNSUPPORTED, "mr_gp_predict: the two-kernel path needs proj_rows in multiples of %d", MR_GP_PAD);
    if (gp->proj_rows > 0 && !fused_spectral_disabled()) {
        // spectral form: one fused kernel, no K_q workspace
        if ((uintptr_t)gp->linv & 15u) return fail(MR_ERR_ARG, "mr_gp_predict: projection must be 16-byte aligned");
        const unsigned blocks = (unsigned)((n_q + GP_BM - 1) / GP_BM);
        const int nt = gp->proj_rows >= MR_GP_PAD ? 4 : gp->proj_rows / 32;
        auto launch = [&](auto kernel) {
            cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDmmaSmemBytes);
            kernel<<<blocks, 256, kDmmaSmemBytes, s>>>(q, n_q, gp->x_train_scaled, gp->alpha, gp->linv, gp->n_pad, gp->proj_rows,
                                                       gp->length_scale, 1.0 + gp->noise_level, mean, std);
        };
        if (gp->dim == 1) {
            if (nt == 4) launch(gp_posterior_spectral_kernel<1, 4>); else if (nt == 3) launch(gp_posterior_spectral_kernel<1, 3>);
            else if (nt == 2) launch(gp_posterior_spectral_kernel<1, 2>); else launch(gp_posterior_spectral_kernel<1, 1>);
        } else {
            if (nt == 4) launch(gp_posterior_spectral_kernel<2, 4>); else if (nt == 3) launch(gp_posterior_spectral_kernel<2, 3>);
            else if (nt == 2) launch(gp_posterior_spectral_kernel<2, 2>); else launch(gp_posterior_spectral_kernel<2, 1>);
        }
        return check_launch("mr_gp_predict(spectral)");
    }
    if (!workspace || workspace_bytes < mr_gp_workspace_bytes(gp, n_q, 1))
        return fail(MR_ERR_ARG, "mr_gp_predict: workspace too small (%lld < %lld)", (long long)workspace_bytes,
                    (long long)mr_gp_workspace_bytes(gp, n_q, 1));
    if (((uintptr_t)workspace & 15u) || ((uintptr_t)gp->linv & 15u))
        return fail(MR_ERR_ARG, "mr_gp_predict: workspace / linv must be 16-byte aligned");
    const int64_t chunk_cap = round_up(n_q < kGpChunk ? n_q : kGpChunk, GP_BM);
    double* kq = (double*)workspace;
    double* ssq = kq + chunk_cap * gp->n_pad;
    const size_t smem = kDmmaSmemBytes;
    cudaFuncSetAttribute(gp_var_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    for (int64_t q0 = 0; q0 < n_q; q0 += kGpChunk) {
        const int64_t nq = (n_q - q0) < kGpChunk ? (n_q - q0) : kGpChunk;
        const int64_t nq_pad = round_up(nq, GP_BM);
        if (nq_pad > nq) cudaMemsetAsync(kq + nq * gp->n_pad, 0, (size_t)(nq_pad - nq) * gp->n_pad * 8, s);
        if (gp->dim == 1) launch_kq_mean<1, true>(q + q0, nq, gp, kq, mean + q0, s);
        else launch_kq_mean<2, true>(q + q0 * 2, nq, gp, kq, mean + q0, s);
        cudaMemsetAsync(ssq, 0, (size_t)nq_pad * 8, s);
        const int rows = gp->proj_rows > 0 ? gp->proj_rows : gp->n_pad;
        dim3 grid((unsigned)(nq_pad / GP_BM), (unsigned)(rows / GP_BN));
        gp_var_kernel<<<grid, 256, smem, s>>>(kq, gp->linv, gp->n_pad, nq_pad, ssq, gp->proj_rows > 0 ? 1 : 0);
        gp_std_finish_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(ssq, nq, 1.0 + gp->noise_level, std + q0);
        int rc = check_launch("mr_gp_predict");
        if (rc) return rc;
    }
    return MR_OK;
}


int mr_gp_correct_heading(const mr_gp_model* gpx, const mr_gp_model* gpy, const double* vd, int64_t n, double a0,
                          double freq, double drift_x, double drift_y, double* alpha_out, int32_t* nfev_out, void* stream) {
    mr::NvtxRange nvtx_range("mr_gp_correct_heading");
    using namespace mr;
    if (!gpx || !gpy || !gpx->x_train_scaled || !gpy->x_train_scaled || !gpx->alpha || !gpy->alpha)
        return fail(MR_ERR_ARG, "mr_gp_correct_heading: null model");
    if (gpx->dim != 1 || gpy->dim != 1) return fail(MR_ERR_UNSUPPORTED, "mr_gp_correct_heading: heading GPs have dim 1");
    if (gpx->n_pad != gpy->n_pad || gpx->n_train != gpy->n_train)
        return fail(MR_ERR_ARG, "mr_gp_correct_heading: the two GPs must share their training inputs");
    if (n < 0) return fail(MR_ERR_ARG, "mr_gp_correct_heading: bad n");
    if (n == 0) return MR_OK;
    if (!vd || !alpha_out) return fail(MR_ERR_ARG, "mr_gp_correct_heading: null vd/alpha_out");
    HeadingProblem hp{a0 * freq, drift_x, drift_y};
    const int threads = 256;
    const unsigned blocks = (unsigned)((n * 32 + threads - 1) / threads);
    gp_correct_heading_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(
        vd, n, hp, gpx->x_train_scaled, gpx->alpha, gpx->length_scale, gpy->x_train_scaled, gpy->alpha, gpy->length_scale,
        gpx->n_pad, gpx->n_train, -3.141592653589793, 3.141592653589793, 1e-5, 500, alpha_out, nfev_out);
    return check_launch("mr_gp_correct_heading");
}

int mr_gp_correct_heading_cheb(const double* coef_x, const double* coef_y, int32_t n_coef, const double* vd, int64_t n,
                               double a0, double freq, double drift_x, double drift_y, double* alpha_out, int32_t* nfev_out,
                               void* stream) {
    mr::NvtxRange nvtx_range("mr_gp_correct_heading_cheb");
    using namespace mr;
    if (!coef_x || !coef_y) return fail(MR_ERR_ARG, "mr_gp_correct_heading_cheb: null coefficients");
    if (n_coef < 1 || n_coef > 4096) return fail(MR_ERR_ARG, "mr_gp_correct_heading_cheb: need 1 <= n_coef <= 4096");
    if (n < 0) return fail(MR_ERR_ARG, "mr_gp_correct_heading_cheb: bad n");
    if (n == 0) return MR_OK;
    if (!vd || !alpha_out) return fail(MR_ERR_ARG, "mr_gp_correct_heading_cheb: null vd/alpha_out");
    HeadingProblem hp{a0 * freq, drift_x, drift_y};
    const size_t smem = (size_t)n_coef * 2 * sizeof(double);
    if (smem > 48 * 1024) cudaFuncSetAttribute(gp_correct_heading_cheb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const unsigned blocks = (unsigned)((n + 127) / 128);
    gp_correct_heading_cheb_kernel<<<blocks, 128, smem, (cudaStream_t)stream>>>(vd, n, hp, coef_x, coef_y, n_coef, -3.141592653589793,
                                                                               3.141592653589793, 1e-5, 500, alpha_out, nfev_out);
    return check_launch("mr_gp_correct_heading_cheb");
}

int mr_gp_correct_action_2d(const mr_gp_model* gpx, const mr_gp_model* gpy, const double* vd, int64_t n, double a0,
                            const double lo[2], const double hi[2], double* x_out, int32_t* iters_out, uint8_t* status_out,
                            void* stream) {
    mr::NvtxRange nvtx_range("mr_gp_correct_action_2d");
    using namespace mr;
    if (!gpx || !gpy || !gpx->x_train_scaled || !gpy->x_train_scaled || !gpx->alpha || !gpy->alpha)
        return fail(MR_ERR_ARG, "mr_gp_correct_action_2d: null model");
    if (gpx->dim != 2 || gpy->dim != 2) return fail(MR_ERR_UNSUPPORTED, "mr_gp_correct_action_2d: (alpha, f) GPs have dim 2");
    if (gpx->n_pad != gpy->n_pad || gpx->n_train != gpy->n_train)
        return fail(MR_ERR_ARG, "mr_gp_correct_action_2d: the two GPs must share their training inputs");
    if (gpx->n_train <= 0 || gpx->n_train > gpx->n_pad || !(gpx->length_scale > 0) || !(gpy->length_scale > 0))
        return fail(MR_ERR_ARG, "mr_gp_correct_action_2d: bad n_train / length_scale");
    if (n < 0) return fail(MR_ERR_ARG, "mr_gp_correct_action_2d: bad n");
    if (n == 0) return MR_OK;
    if (!vd || !x_out) return fail(MR_ERR_ARG, "mr_gp_correct_action_2d: null vd/x_out");
    if (!lo || !hi) return fail(MR_ERR_ARG, "mr_gp_correct_action_2d: null bounds");
    for (int c = 0; c < 2; ++c)
        if (!std::isfinite(lo[c]) || !std::isfinite(hi[c]) || !(lo[c] < hi[c]))
            return fail(MR_ERR_ARG, "mr_gp_correct_action_2d: bounds must be finite with lo < hi");
    if (!std::isfinite(a0) || !(a0 > 0)) return fail(MR_ERR_ARG, "mr_gp_correct_action_2d: a0 must be finite and > 0");
    const int threads = 256;
    const unsigned blocks = (unsigned)((n * 32 + threads - 1) / threads);
    gp_correct_action_2d_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(
        vd, n, a0, gpx->x_train_scaled, gpx->alpha, gpx->length_scale, gpy->x_train_scaled, gpy->alpha, gpy->length_scale,
        gpx->n_train, lo[0], lo[1], hi[0], hi[1], x_out, iters_out, status_out);
    return check_launch("mr_gp_correct_action_2d");
}

int32_t mr_actor_param_count(void) { return mr::kActorParams; }

int mr_actor_forward(const float* actor, const void* obs, int64_t obs_row_stride, int64_t n, int32_t dtype,
                     const double action_high[2], void* actions, void* stream) {
    mr::NvtxRange nvtx_range("mr_actor_forward");
    using namespace mr;
    if (!actor || !obs || !actions || !action_high) return fail(MR_ERR_ARG, "mr_actor_forward: null argument");
    if (n < 0) return fail(MR_ERR_ARG, "mr_actor_forward: bad n");
    if (n == 0) return MR_OK;
    const int threads = 128;
    const unsigned blocks = (unsigned)((n + threads - 1) / threads);
    const size_t smem = kActorParams * sizeof(float);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t stride = obs_row_stride ? obs_row_stride : n;
    if (dtype == MR_F64)
        actor_forward_kernel<double><<<blocks, threads, smem, s>>>(actor, (const double*)obs, stride, n, (float)action_high[0], (float)action_high[1], (double*)actions);
    else if (dtype == MR_F32)
        actor_forward_kernel<float><<<blocks, threads, smem, s>>>(actor, (const float*)obs, stride, n, (float)action_high[0], (float)action_high[1], (float*)actions);
    else return fail(MR_ERR_ARG, "mr_actor_forward: bad dtype");
    return check_launch("mr_actor_forward");
}

int mr_actor_forward_env(const float* actor, const void* obs, int64_t obs_row_stride, int64_t n, int32_t dtype,
                         const double action_high[2], void* actions, void* stream) {
    mr::NvtxRange nvtx_range("mr_actor_forward_env");
    using namespace mr;
    if (!actor || !obs || !actions || !action_high) return fail(MR_ERR_ARG, "mr_actor_forward_env: null argument");
    if (n < 0) return fail(MR_ERR_ARG, "mr_actor_forward_env: bad n");
    if (n == 0) return MR_OK;
    if (dtype != MR_F64 && dtype != MR_F32) return fail(MR_ERR_ARG, "mr_actor_forward_env: bad dtype");
    static int ctas[kMaxDevices] = {};
    const int dev = current_device();
    if (!ctas[dev]) {
        cudaFuncSetAttribute(actor_forward_tc_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ActorTcSmem));
        cudaFuncSetAttribute(actor_forward_tc_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ActorTcSmem));
        int sms = 0, occ = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, actor_forward_tc_kernel<double>, kTcRows, sizeof(ActorTcSmem));
        ctas[dev] = (sms > 0 ? sms : 148) * (occ > 0 ? occ : 1);
    }
    const int64_t tiles = (n + kTcRows - 1) / kTcRows;
    const unsigned grid = (unsigned)(tiles < ctas[dev] ? tiles : ctas[dev]);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t stride = obs_row_stride ? obs_row_stride : n;
    if (dtype == MR_F64)
        actor_forward_tc_kernel<double><<<grid, kTcRows, sizeof(ActorTcSmem), s>>>(actor, (const double*)obs, stride, n, (float)action_high[0], (float)action_high[1], (double*)actions);
    else
        actor_forward_tc_kernel<float><<<grid, kTcRows, sizeof(ActorTcSmem), s>>>(actor, (const float*)obs, stride, n, (float)action_high[0], (float)action_high[1], (float*)actions);
    return check_launch("mr_actor_forward_env");
}

}  // extern "C"
