// DDPG learner on the device (RL/MR_ddpg.py:16-78 replay / OU noise, :80-231 networks, :285-305 update block;
// SURVEY §8f rank 3): replay ring in HBM, and ONE kernel launch per learner update — sampling, target networks,
// critic forward/backward + Adam, action gradient, actor backward + Adam, soft target updates.
//
// The networks are tiny (5-64-64-2 and 5-64-(+2)-32-1) and the reference batch is 64, so an update is latency
// bound, not throughput bound: one CTA keeps a 64-sample tile of every activation in shared memory and walks
// the phases with CTA barriers; the networks a phase reads are staged in shared memory (44 KB).  Larger batches loop over
// 64-sample tiles and accumulate the weight gradients; above 256 samples a data-parallel variant (one CTA per SM, see
// below) takes over.  fp32 throughout, like the reference's TensorFlow graph.
//
// Batch norm: the reference never switches tflearn into training mode, so batch_normalization is the inference
// transform gamma * (x - moving_mean) / sqrt(moving_var + 1e-5) + beta with trainable gamma / beta and frozen
// moving statistics (oracle/ddpg_oracle.py states this; parity unpinned — no TensorFlow in this image).
#include <cuda_runtime.h>

#include <cmath>
#include <initializer_list>

#include "mr_actor.cuh"
#include "mr_common.cuh"
#include "mr_ou.cuh"

namespace mr {

// packed critic layout (float32, input-major matrices)
constexpr int kC_Wc1 = 0;                                   // [5][64]
constexpr int kC_Bc1 = kC_Wc1 + 5 * 64;
constexpr int kC_Gc = kC_Bc1 + 64;
constexpr int kC_Bec = kC_Gc + 64;
constexpr int kC_Mc = kC_Bec + 64;                          // moving mean / variance: not trainable
constexpr int kC_Vc = kC_Mc + 64;
constexpr int kC_T1 = kC_Vc + 64;                           // [64][32]
constexpr int kC_T1b = kC_T1 + 64 * 32;                     // created by the reference, never used in its graph
constexpr int kC_T2 = kC_T1b + 32;                          // [2][32]
constexpr int kC_T2b = kC_T2 + 2 * 32;
constexpr int kC_Wo = kC_T2b + 32;                          // [32]
constexpr int kC_Bo = kC_Wo + 32;
constexpr int kCriticParams = kC_Bo + 1;                    // 2849 floats

constexpr int kTile = 64;                                   // samples per shared-memory tile
constexpr int kLd64 = 65, kLd32 = 33;                       // padded rows: lanes over samples hit distinct banks
constexpr int kMaxBatch = 4096;                             // single-CTA kernel (indices live in shared memory)
constexpr int kWideBatch = 64;                              // above one tile the data-parallel kernels take over (if a workspace is
                                                            // given): measured 296 us single-CTA vs ~80 us at 256 samples
constexpr int kMaxCtas = 256;
#ifndef MR_DDPG_THREADS
#define MR_DDPG_THREADS 1024                                // one CTA; the phases are short loops over <= 4160 work items
#endif
constexpr int kDdpgThreads = MR_DDPG_THREADS;

struct DdpgHyper { float gamma, tau, lr_actor, lr_critic, bound0, bound1, beta1, beta2, eps; };

struct DdpgSmem {
    float S[kTile * 5], S2[kTile * 5], A[kTile * 2], A2[kTile * 2], R[kTile], D[kTile], Y[kTile], Q[kTile], DQ[kTile];
    float T[kTile * 2], DU[kTile * 2];
    float Z1[kTile * kLd64], H1[kTile * kLd64], Z2[kTile * kLd64], H2[kTile * kLd64];
    float ZC[kTile * kLd64], C1[kTile * kLd64], G1[kTile * kLd64], G2[kTile * kLd64];
    float C2[kTile * kLd32], GC2[kTile * kLd32];
    // the networks the current phase reads: L2 latency on every weight would otherwise dominate these short loops
    alignas(16) float wA[kActorParams + 2];                  // target actor (critic phase), then the online actor
    alignas(16) float wC[kCriticParams + 3];                 // online critic (kept in step with Adam's writes)
    alignas(16) float wCt[kCriticParams + 3];                // target critic
    int idx[kMaxBatch];
};

__device__ void load_weights(float* dst, const float* src, int n) {
    for (int k = threadIdx.x; k < n; k += blockDim.x) dst[k] = src[k];
    __syncthreads();
}

// ---- dense layers on shared-memory tiles; every helper is called by the whole CTA and ends with a barrier ----------
// (weight pointers are deliberately NOT __restrict__/read-only here: Adam rewrites them between phases of one launch)
// Every thread owns a small register tile so that each shared-memory load feeds two or four FMAs (the phases are
// load-issue bound otherwise: ncu showed 35 % LDS against 20 % FFMA with one output per thread).
// Y[s][j] = (acc ? Y[s][j] : b[j]) + sum_i X[s][i] W[i][j]       2 samples x 2 adjacent outputs per thread; `out` even
__device__ void fc_fwd(const float* X, int ldx, int nb, int in, const float* W, const float* b,
                       int out, float* Y, int ldy, bool acc) {
    const int hp = out >> 1;
    for (int e = threadIdx.x; e < ((nb + 1) >> 1) * hp; e += blockDim.x) {
        const int sp = e / hp, j = 2 * (e - sp * hp), s0 = 2 * sp, s1 = s0 + 1;     // row s1 == nb is scratch, never stored
        float a00, a01, a10, a11;
        if (acc) { a00 = Y[s0 * ldy + j]; a01 = Y[s0 * ldy + j + 1]; a10 = Y[s1 * ldy + j]; a11 = Y[s1 * ldy + j + 1]; }
        else { a00 = a10 = b ? b[j] : 0.f; a01 = a11 = b ? b[j + 1] : 0.f; }
        const float* x0 = X + s0 * ldx;
        const float* x1 = X + s1 * ldx;
#pragma unroll 4
        for (int i = 0; i < in; ++i) {
            const float2 w = *reinterpret_cast<const float2*>(W + i * out + j);
            const float u0 = x0[i], u1 = x1[i];
            a00 = fmaf(u0, w.x, a00); a01 = fmaf(u0, w.y, a01);
            a10 = fmaf(u1, w.x, a10); a11 = fmaf(u1, w.y, a11);
        }
        Y[s0 * ldy + j] = a00; Y[s0 * ldy + j + 1] = a01;
        if (s1 < nb) { Y[s1 * ldy + j] = a10; Y[s1 * ldy + j + 1] = a11; }
    }
    __syncthreads();
}
// H = relu(gamma (Z - mean) rsqrt(var + eps) + beta)
__device__ void bn_relu_fwd(const float* Z, float* H, int nb, const float* g, const float* be,
                            const float* m, const float* v) {
    for (int e = threadIdx.x; e < nb * 64; e += blockDim.x) {
        const int s = e >> 6, j = e & 63;
        const float y = g[j] * (Z[s * kLd64 + j] - m[j]) * (1.0f / sqrtf(v[j] + kBnEps)) + be[j];
        H[s * kLd64 + j] = y > 0.f ? y : 0.f;
    }
    __syncthreads();
}
// dX[s][i] = sum_j dY[s][j] W[i][j]                              lanes over s (W broadcast, dY rows padded); 4 inputs per thread
__device__ void fc_bwd_x(const float* dY, int ldy, int nb, int out, const float* W, int in, float* dX, int ldx) {
    if ((in & 3) == 0) {
        for (int e = threadIdx.x; e < nb * (in >> 2); e += blockDim.x) {
            const int ig = e / nb, s = e - ig * nb, i0 = 4 * ig;
            const float* w = W + i0 * out;
            float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
#pragma unroll 4
            for (int j = 0; j < out; ++j) {
                const float d = dY[s * ldy + j];
                v0 = fmaf(d, w[j], v0); v1 = fmaf(d, w[out + j], v1); v2 = fmaf(d, w[2 * out + j], v2); v3 = fmaf(d, w[3 * out + j], v3);
            }
            float* dst = dX + s * ldx + i0;
            dst[0] = v0; dst[1] = v1; dst[2] = v2; dst[3] = v3;
        }
    } else {
        for (int e = threadIdx.x; e < nb * in; e += blockDim.x) {
            const int i = e / nb, s = e - i * nb;
            float v = 0.f;
            for (int j = 0; j < out; ++j) v = fmaf(dY[s * ldy + j], W[i * out + j], v);
            dX[s * ldx + i] = v;
        }
    }
    __syncthreads();
}
// gW[i][j] (+)= sum_s X[s][i] dY[s][j];  gb[j] (+)= sum_s dY[s][j] (the bias is row `in` with x = 1)
// 2 rows x 2 columns (j, j + out/2: conflict-free) per thread; `out` even
__device__ void fc_bwd_w(const float* X, int ldx, const float* dY, int ldy, int nb, int in, int out, float* gW,
                         float* gb, bool acc) {
    const int hp = out >> 1, rows = in + 1;
    for (int e = threadIdx.x; e < ((rows + 1) >> 1) * hp; e += blockDim.x) {
        const int rp = e / hp, j0 = e - rp * hp, j1 = j0 + hp, r0 = 2 * rp, r1 = r0 + 1;
        float v00 = 0.f, v01 = 0.f, v10 = 0.f, v11 = 0.f;
        const bool x0one = r0 == in, x1one = r1 >= in;            // bias row (or the unused row past it)
        const float* c0 = X + (x0one ? 0 : r0);
        const float* c1 = X + (x1one ? 0 : r1);
#pragma unroll 4
        for (int s = 0; s < nb; ++s) {
            const float d0 = dY[s * ldy + j0], d1 = dY[s * ldy + j1];
            const float u0 = x0one ? 1.f : c0[s * ldx], u1 = x1one ? 1.f : c1[s * ldx];
            v00 = fmaf(u0, d0, v00); v01 = fmaf(u0, d1, v01);
            v10 = fmaf(u1, d0, v10); v11 = fmaf(u1, d1, v11);
        }
        float* d0p = r0 < in ? gW + r0 * out : gb;                // gb may be null (t1's bias is not in the graph)
        if (d0p) { d0p[j0] = acc ? d0p[j0] + v00 : v00; d0p[j1] = acc ? d0p[j1] + v01 : v01; }
        if (r1 <= in) {
            float* d1p = r1 < in ? gW + r1 * out : gb;
            if (d1p) { d1p[j0] = acc ? d1p[j0] + v10 : v10; d1p[j1] = acc ? d1p[j1] + v11 : v11; }
        }
    }
    __syncthreads();
}
// batch norm + relu backward, in place on G (incoming dL/dH): G <- dL/dZ; ggamma, gbeta (+)=
__device__ void bn_relu_bwd(float* G, const float* Z, const float* H, int nb, const float* g,
                            const float* m, const float* v, float* gg,
                            float* gbe, bool acc) {
    for (int e = threadIdx.x; e < nb * 64; e += blockDim.x) {
        const int s = e >> 6, j = e & 63;
        if (!(H[s * kLd64 + j] > 0.f)) G[s * kLd64 + j] = 0.f;
    }
    __syncthreads();
    if (threadIdx.x < 64) {
        const int j = threadIdx.x;
        const float rs = 1.0f / sqrtf(v[j] + kBnEps);
        float a = 0.f, b = 0.f;
        for (int s = 0; s < nb; ++s) { const float d = G[s * kLd64 + j]; a = fmaf(d, (Z[s * kLd64 + j] - m[j]) * rs, a); b += d; }
        gg[j] = acc ? gg[j] + a : a;
        gbe[j] = acc ? gbe[j] + b : b;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nb * 64; e += blockDim.x) {
        const int s = e >> 6, j = e & 63;
        G[s * kLd64 + j] *= g[j] * (1.0f / sqrtf(v[j] + kBnEps));
    }
    __syncthreads();
}

__device__ void actor_fwd_tile(DdpgSmem& sm, const float* X, int nb, const float* w, float b0, float b1, float* Aout) {
    fc_fwd(X, 5, nb, 5, w + kOffW1, w + kOffB1, 64, sm.Z1, kLd64, false);
    bn_relu_fwd(sm.Z1, sm.H1, nb, w + kOffG1, w + kOffBe1, w + kOffM1, w + kOffV1);
    fc_fwd(sm.H1, kLd64, nb, 64, w + kOffW2, w + kOffB2, 64, sm.Z2, kLd64, false);
    bn_relu_fwd(sm.Z2, sm.H2, nb, w + kOffG2, w + kOffBe2, w + kOffM2, w + kOffV2);
    fc_fwd(sm.H2, kLd64, nb, 64, w + kOffW3, w + kOffB3, 2, sm.T, 2, false);
    for (int e = threadIdx.x; e < nb * 2; e += blockDim.x) {
        const float t = tanhf(sm.T[e]);
        sm.T[e] = t;
        Aout[e] = t * ((e & 1) ? b1 : b0);
    }
    __syncthreads();
}

__device__ void critic_fwd_tile(DdpgSmem& sm, const float* X, const float* Act, int nb, const float* c, float* Qout) {
    fc_fwd(X, 5, nb, 5, c + kC_Wc1, c + kC_Bc1, 64, sm.ZC, kLd64, false);
    bn_relu_fwd(sm.ZC, sm.C1, nb, c + kC_Gc, c + kC_Bec, c + kC_Mc, c + kC_Vc);
    fc_fwd(sm.C1, kLd64, nb, 64, c + kC_T1, c + kC_T2b, 32, sm.C2, kLd32, false);      // + t2.b, as the reference's graph
    fc_fwd(Act, 2, nb, 2, c + kC_T2, nullptr, 32, sm.C2, kLd32, true);
    for (int e = threadIdx.x; e < nb * 32; e += blockDim.x) {
        const int s = e >> 5, j = e & 31;
        const float y = sm.C2[s * kLd32 + j];
        sm.C2[s * kLd32 + j] = y > 0.f ? y : 0.f;
    }
    __syncthreads();
    if (Qout) {
        for (int s = threadIdx.x; s < nb; s += blockDim.x) {
            float q = c[kC_Bo];
            for (int j = 0; j < 32; ++j) q = fmaf(sm.C2[s * kLd32 + j], c[kC_Wo + j], q);
            Qout[s] = q;
        }
        __syncthreads();
    }
}

// TF1 AdamOptimizer: lr_t = lr sqrt(1 - b2^t) / (1 - b1^t);  theta -= lr_t m / (sqrt(v) + eps)
__device__ void adam_step(float* p, float* p_smem, const float* g, float* m, float* v, int n,
                          int frozen_lo0, int frozen_hi0, int frozen_lo1, int frozen_hi1, float lr_t, const DdpgHyper& h) {
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
        if ((k >= frozen_lo0 && k < frozen_hi0) || (k >= frozen_lo1 && k < frozen_hi1)) continue;
        const float gk = g[k];
        const float mk = h.beta1 * m[k] + (1.f - h.beta1) * gk;
        const float vk = h.beta2 * v[k] + (1.f - h.beta2) * gk * gk;
        m[k] = mk; v[k] = vk;
        const float pk = p[k] - lr_t * mk / (sqrtf(vk) + h.eps);
        p[k] = pk;
        if (p_smem) p_smem[k] = pk;
    }
    __syncthreads();
}

__device__ void gather_tile(DdpgSmem& sm, int t0, int nb, const float* rs, const float* ra,
                            const float* rr, const float* rd, const float* rs2) {
    for (int e = threadIdx.x; e < nb * 5; e += blockDim.x) {
        const int s = e / 5, k = e - s * 5;
        const int64_t row = sm.idx[t0 + s];
        sm.S[e] = rs[row * 5 + k];
        sm.S2[e] = rs2[row * 5 + k];
    }
    for (int e = threadIdx.x; e < nb * 2; e += blockDim.x) sm.A[e] = ra[(int64_t)sm.idx[t0 + (e >> 1)] * 2 + (e & 1)];
    for (int s = threadIdx.x; s < nb; s += blockDim.x) { sm.R[s] = rr[sm.idx[t0 + s]]; sm.D[s] = rd[sm.idx[t0 + s]]; }
    __syncthreads();
}

// ---- one 64-sample tile of the critic step: y = r + gamma Q'(s2, mu'(s2)) (1 - done); d/dtheta of mean (y - Q(s, a))^2 -----
// expects the tile gathered in sm.S/A/R/D/S2 and sm.wA = target actor, sm.wCt = target critic, sm.wC = online critic
__device__ void critic_tile(DdpgSmem& sm, int nb, bool acc, float inv_b, const DdpgHyper& h, float* gc, float& loss_acc, float& q_acc) {
    const int tid = threadIdx.x;
    actor_fwd_tile(sm, sm.S2, nb, sm.wA, h.bound0, h.bound1, sm.A2);
    critic_fwd_tile(sm, sm.S2, sm.A2, nb, sm.wCt, sm.Q);
    for (int s = tid; s < nb; s += blockDim.x) sm.Y[s] = sm.R[s] + h.gamma * sm.Q[s] * (1.f - sm.D[s]);
    __syncthreads();
    critic_fwd_tile(sm, sm.S, sm.A, nb, sm.wC, sm.Q);
    for (int s = tid; s < nb; s += blockDim.x) sm.DQ[s] = 2.f * (sm.Q[s] - sm.Y[s]) * inv_b;
    __syncthreads();
    if (tid == 0) for (int s = 0; s < nb; ++s) { const float e = sm.Y[s] - sm.Q[s]; loss_acc += e * e; q_acc += sm.Q[s]; }
    // output layer: gWo[j] = sum_s C2[s][j] dQ[s], gbo = sum_s dQ[s];  dC2 = dQ Wo (C2 > 0)
    if (tid < 33) {
        float v = 0.f;
        if (tid < 32) { for (int s = 0; s < nb; ++s) v = fmaf(sm.C2[s * kLd32 + tid], sm.DQ[s], v); }
        else          { for (int s = 0; s < nb; ++s) v += sm.DQ[s]; }
        float* dst = gc + kC_Wo + tid;                    // kC_Bo = kC_Wo + 32
        *dst = acc ? *dst + v : v;
    }
    for (int e = tid; e < nb * 32; e += blockDim.x) {
        const int s = e >> 5, j = e & 31;
        sm.GC2[s * kLd32 + j] = sm.C2[s * kLd32 + j] > 0.f ? sm.DQ[s] * sm.wC[kC_Wo + j] : 0.f;
    }
    __syncthreads();
    fc_bwd_w(sm.C1, kLd64, sm.GC2, kLd32, nb, 64, 32, gc + kC_T1, nullptr, acc);          // t1.b: no gradient
    fc_bwd_w(sm.A, 2, sm.GC2, kLd32, nb, 2, 32, gc + kC_T2, gc + kC_T2b, acc);
    fc_bwd_x(sm.GC2, kLd32, nb, 32, sm.wC + kC_T1, 64, sm.G1, kLd64);
    bn_relu_bwd(sm.G1, sm.ZC, sm.C1, nb, sm.wC + kC_Gc, sm.wC + kC_Mc, sm.wC + kC_Vc, gc + kC_Gc, gc + kC_Bec, acc);
    fc_bwd_w(sm.S, 5, sm.G1, kLd64, nb, 5, 64, gc + kC_Wc1, gc + kC_Bc1, acc);
}

// ---- one tile of the actor step: ascend Q(s, mu(s)) through the critic in sm.wC; d scaled_out/d theta . (-dQ/da) / batch ------
// expects sm.S gathered and sm.wA = online actor
__device__ void actor_tile(DdpgSmem& sm, int nb, bool acc, float inv_b, const DdpgHyper& h, float* ga) {
    const int tid = threadIdx.x;
    actor_fwd_tile(sm, sm.S, nb, sm.wA, h.bound0, h.bound1, sm.A2);          // sm.T keeps tanh(u)
    critic_fwd_tile(sm, sm.S, sm.A2, nb, sm.wC, nullptr);
    for (int e = tid; e < nb * 32; e += blockDim.x) {
        const int s = e >> 5, j = e & 31;
        sm.GC2[s * kLd32 + j] = sm.C2[s * kLd32 + j] > 0.f ? sm.wC[kC_Wo + j] : 0.f;
    }
    __syncthreads();
    fc_bwd_x(sm.GC2, kLd32, nb, 32, sm.wC + kC_T2, 2, sm.DU, 2);             // dQ/da
    for (int e = tid; e < nb * 2; e += blockDim.x) {
        const float th = sm.T[e];
        sm.DU[e] = -sm.DU[e] * inv_b * ((e & 1) ? h.bound1 : h.bound0) * (1.f - th * th);
    }
    __syncthreads();
    fc_bwd_w(sm.H2, kLd64, sm.DU, 2, nb, 64, 2, ga + kOffW3, ga + kOffB3, acc);
    fc_bwd_x(sm.DU, 2, nb, 2, sm.wA + kOffW3, 64, sm.G2, kLd64);
    bn_relu_bwd(sm.G2, sm.Z2, sm.H2, nb, sm.wA + kOffG2, sm.wA + kOffM2, sm.wA + kOffV2, ga + kOffG2, ga + kOffBe2, acc);
    fc_bwd_w(sm.H1, kLd64, sm.G2, kLd64, nb, 64, 64, ga + kOffW2, ga + kOffB2, acc);
    fc_bwd_x(sm.G2, kLd64, nb, 64, sm.wA + kOffW2, 64, sm.G1, kLd64);
    bn_relu_bwd(sm.G1, sm.Z1, sm.H1, nb, sm.wA + kOffG1, sm.wA + kOffM1, sm.wA + kOffV1, ga + kOffG1, ga + kOffBe1, acc);
    fc_bwd_w(sm.S, 5, sm.G1, kLd64, nb, 5, 64, ga + kOffW1, ga + kOffB1, acc);
}

// One learner update by the whole CTA: the body of ddpg_update_kernel (one learner) and of ddpg_update_population_kernel
// (member blockIdx.x of a population).  Member p of a population must compute what the solo kernel computes bit for bit,
// which holds only while ptxas schedules and contracts the float arithmetic of both inlined copies alike: hand the body
// h and keys in registers (as the population kernel does) and check with test_population_update_equals_solo_updates
// (tests/test_ddpg_population.py) after any change here or to the compiler.
__device__ __forceinline__ void ddpg_update_cta(float* __restrict__ actor, float* __restrict__ actor_t, float* __restrict__ critic,
                                                float* __restrict__ critic_t, float* __restrict__ am, float* __restrict__ av,
                                                float* __restrict__ cm, float* __restrict__ cv, float* __restrict__ ga,
                                                float* __restrict__ gc, const float* __restrict__ rs, const float* __restrict__ ra,
                                                const float* __restrict__ rr, const float* __restrict__ rd,
                                                const float* __restrict__ rs2, int64_t count, int batch,
                                                const int64_t* __restrict__ indices, const PhiloxKeys& keys, uint64_t update_index,
                                                const DdpgHyper& h, float* __restrict__ info_out) {
    extern __shared__ __align__(16) unsigned char ddpg_smem_raw[];
    DdpgSmem& sm = *reinterpret_cast<DdpgSmem*>(ddpg_smem_raw);
    const int tid = threadIdx.x;

    // ---- the minibatch: caller-supplied rows, or a uniform sample WITHOUT replacement (random.sample, :43-46) by Floyd's
    //      algorithm, one warp, Philox keyed by (seed; update index, draw)
    if (indices) {
        for (int k = tid; k < batch; k += blockDim.x) sm.idx[k] = (int)indices[k];
    } else {
        for (int t = tid; t < batch; t += blockDim.x) {       // all draws in parallel, then one warp resolves collisions
            uint32_t o0, o1, o2, o3;
            philox4x32_10((uint32_t)t | (4u << 28), (uint32_t)update_index, (uint32_t)(update_index >> 32), 0u, keys.rk, o0, o1, o2, o3);
            const int64_t j = count - batch + t;
            sm.idx[t] = (int)(((uint64_t)o0 * (uint64_t)(j + 1)) >> 32);          // uniform in [0, j]
        }
        __syncthreads();
        if (tid < 32) {
            for (int t = 0; t < batch; ++t) {
                const int cand = sm.idx[t];
                bool hit = false;
                for (int k = tid; k < t; k += 32) hit |= sm.idx[k] == cand;
                if (__any_sync(0xffffffffu, hit) && tid == 0) sm.idx[t] = (int)(count - batch + t);
                __syncwarp();
            }
        }
    }
    __syncthreads();

    load_weights(sm.wA, actor_t, kActorParams);
    load_weights(sm.wCt, critic_t, kCriticParams);
    load_weights(sm.wC, critic, kCriticParams);
    const float inv_b = 1.0f / (float)batch;
    float loss_acc = 0.f, q_acc = 0.f;                         // thread 0 only
    const int n_tiles = (batch + kTile - 1) / kTile;

    // ---- critic: y = r + gamma Q'(s2, mu'(s2)) (1 - done); minimise mean (y - Q(s, a))^2 ------------------------------
    for (int t = 0; t < n_tiles; ++t) {
        const int nb = min(kTile, batch - t * kTile);
        const bool acc = t > 0;
        gather_tile(sm, t * kTile, nb, rs, ra, rr, rd, rs2);
        critic_tile(sm, nb, acc, inv_b, h, gc, loss_acc, q_acc);
    }
    if (tid < 32) gc[kC_T1b + tid] = 0.f;
    __syncthreads();
    {
        const float t = (float)update_index;
        const float lr_t = h.lr_critic * sqrtf(1.f - powf(h.beta2, t)) / (1.f - powf(h.beta1, t));
        adam_step(critic, sm.wC, gc, cm, cv, kCriticParams, kC_Mc, kC_T1, 0, 0, lr_t, h);
    }
    load_weights(sm.wA, actor, kActorParams);

    // ---- actor: ascend Q(s, mu(s)) through the UPDATED critic; gradient = d scaled_out / d theta . (-dQ/da) / batch ------
    for (int t = 0; t < n_tiles; ++t) {
        const int nb = min(kTile, batch - t * kTile);
        const bool acc = t > 0;
        gather_tile(sm, t * kTile, nb, rs, ra, rr, rd, rs2);
        actor_tile(sm, nb, acc, inv_b, h, ga);
    }
    {
        const float t = (float)update_index;
        const float lr_t = h.lr_actor * sqrtf(1.f - powf(h.beta2, t)) / (1.f - powf(h.beta1, t));
        adam_step(actor, nullptr, ga, am, av, kActorParams, kOffM1, kOffW2, kOffM2, kOffW3, lr_t, h);
    }

    // ---- soft target updates over the trainable variables (:98-103, :183-188) -----------------------------------------------
    for (int k = tid; k < kActorParams; k += blockDim.x) {
        if ((k >= kOffM1 && k < kOffW2) || (k >= kOffM2 && k < kOffW3)) continue;
        actor_t[k] = h.tau * actor[k] + (1.f - h.tau) * actor_t[k];
    }
    for (int k = tid; k < kCriticParams; k += blockDim.x) {
        if (k >= kC_Mc && k < kC_T1) continue;
        critic_t[k] = h.tau * critic[k] + (1.f - h.tau) * critic_t[k];
    }
    if (tid == 0 && info_out) { info_out[0] = loss_acc * inv_b; info_out[1] = q_acc * inv_b; }
}

__global__ void __launch_bounds__(kDdpgThreads, 1)
ddpg_update_kernel(float* __restrict__ actor, float* __restrict__ actor_t, float* __restrict__ critic, float* __restrict__ critic_t,
                   float* __restrict__ am, float* __restrict__ av, float* __restrict__ cm, float* __restrict__ cv,
                   float* __restrict__ ga, float* __restrict__ gc,
                   const float* __restrict__ rs, const float* __restrict__ ra, const float* __restrict__ rr,
                   const float* __restrict__ rd, const float* __restrict__ rs2, int64_t count, int batch,
                   const int64_t* __restrict__ indices, PhiloxKeys keys, uint64_t update_index, DdpgHyper h,
                   float* __restrict__ info_out) {
    ddpg_update_cta(actor, actor_t, critic, critic_t, am, av, cm, cv, ga, gc, rs, ra, rr, rd, rs2, count, batch, indices, keys,
                    update_index, h, info_out);
}

// ---- a population of independent learners (mr_ddpg_update_population): one CTA per member, every array member-major.
//      The members' hyper-parameters and sampling keys travel in the launch's parameter space (no device buffer, no copy).
constexpr int kMaxMembers = MR_DDPG_MAX_MEMBERS;
struct DdpgMember { DdpgHyper h; PhiloxKeys keys; };
struct DdpgMembers { DdpgMember m[kMaxMembers]; };             // 29.7 KB: kernel parameters may take 32 KB (CUDA 12.1+)
static_assert(sizeof(DdpgMembers) < 31 * 1024, "the members must fit the kernel parameter space next to the pointers");
struct DdpgStack {                                              // mr_ddpg_state + mr_replay of the population
    float *actor, *actor_t, *critic, *critic_t, *am, *av, *cm, *cv, *ga, *gc;
    const float *rs, *ra, *rr, *rd, *rs2;
    int64_t capacity;
};

__global__ void __launch_bounds__(kDdpgThreads, 1)
ddpg_update_population_kernel(DdpgStack ps, int64_t count, int batch, uint64_t update_index, float* __restrict__ info_out,
                              const __grid_constant__ DdpgMembers mem) {
    const int64_t p = blockIdx.x, pa = p * kActorParams, pc = p * kCriticParams, row = p * ps.capacity;
    const DdpgHyper h = mem.m[p].h;                              // in registers, as the solo kernel's parameters: the
    const PhiloxKeys keys = mem.m[p].keys;                       // compiler then hoists and contracts the same way
    ddpg_update_cta(ps.actor + pa, ps.actor_t + pa, ps.critic + pc, ps.critic_t + pc, ps.am + pa, ps.av + pa, ps.cm + pc,
                    ps.cv + pc, ps.ga + pa, ps.gc + pc, ps.rs + row * 5, ps.ra + row * 2, ps.rr + row, ps.rd + row,
                    ps.rs2 + row * 5, count, batch, nullptr, keys, update_index, h, info_out ? info_out + 2 * p : nullptr);
}

// =====================================================================================================================
// Large minibatches: the same update, data-parallel over CTAs (one per SM).  Every CTA walks its share of the 64-sample
// tiles and leaves its partial weight gradients in its own slab; a second kernel adds the slabs in a fixed order
// (deterministic), applies Adam and the soft target update.  critic grads -> critic Adam -> actor grads (through the
// updated critic) -> actor Adam: four launches instead of one, but 148x the arithmetic throughput.
// =====================================================================================================================
constexpr int kSlab = 5248;                                  // floats per CTA slab: >= max(kActorParams, kCriticParams) + 2

__device__ void tile_indices(DdpgSmem& sm, const int64_t* idx, int t0, int nb) {
    for (int k = threadIdx.x; k < nb; k += blockDim.x) sm.idx[k] = (int)idx[t0 + k];
    __syncthreads();
}

__global__ void __launch_bounds__(kDdpgThreads, 1)
ddpg_critic_grad_kernel(const float* __restrict__ actor_t, const float* __restrict__ critic, const float* __restrict__ critic_t,
                        const float* __restrict__ rs, const float* __restrict__ ra, const float* __restrict__ rr,
                        const float* __restrict__ rd, const float* __restrict__ rs2, const int64_t* __restrict__ idx,
                        int batch, DdpgHyper h, float* __restrict__ slabs) {
    extern __shared__ __align__(16) unsigned char ddpg_smem_raw[];
    DdpgSmem& sm = *reinterpret_cast<DdpgSmem*>(ddpg_smem_raw);
    load_weights(sm.wA, actor_t, kActorParams);
    load_weights(sm.wCt, critic_t, kCriticParams);
    load_weights(sm.wC, critic, kCriticParams);
    float* gc = slabs + (int64_t)blockIdx.x * kSlab;
    const float inv_b = 1.0f / (float)batch;
    float loss_acc = 0.f, q_acc = 0.f;
    const int n_tiles = (batch + kTile - 1) / kTile;
    bool acc = false;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, acc = true) {
        const int nb = min(kTile, batch - t * kTile);
        tile_indices(sm, idx, t * kTile, nb);
        gather_tile(sm, 0, nb, rs, ra, rr, rd, rs2);
        critic_tile(sm, nb, acc, inv_b, h, gc, loss_acc, q_acc);
    }
    if (threadIdx.x < 32) gc[kC_T1b + threadIdx.x] = 0.f;
    if (threadIdx.x >= 64 && threadIdx.x < 128) { gc[kC_Mc + threadIdx.x - 64] = 0.f; gc[kC_Vc + threadIdx.x - 64] = 0.f; }
    if (threadIdx.x == 0) { gc[kCriticParams] = loss_acc; gc[kCriticParams + 1] = q_acc; }
}

__global__ void __launch_bounds__(kDdpgThreads, 1)
ddpg_actor_grad_kernel(const float* __restrict__ actor, const float* __restrict__ critic,
                       const float* __restrict__ rs, const float* __restrict__ ra, const float* __restrict__ rr,
                       const float* __restrict__ rd, const float* __restrict__ rs2, const int64_t* __restrict__ idx,
                       int batch, DdpgHyper h, float* __restrict__ slabs) {
    extern __shared__ __align__(16) unsigned char ddpg_smem_raw[];
    DdpgSmem& sm = *reinterpret_cast<DdpgSmem*>(ddpg_smem_raw);
    load_weights(sm.wA, actor, kActorParams);
    load_weights(sm.wC, critic, kCriticParams);
    float* ga = slabs + (int64_t)blockIdx.x * kSlab;
    const float inv_b = 1.0f / (float)batch;
    const int n_tiles = (batch + kTile - 1) / kTile;
    bool acc = false;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, acc = true) {
        const int nb = min(kTile, batch - t * kTile);
        tile_indices(sm, idx, t * kTile, nb);
        gather_tile(sm, 0, nb, rs, ra, rr, rd, rs2);
        actor_tile(sm, nb, acc, inv_b, h, ga);
    }
}

// sum the CTA slabs in order, TF1 Adam, soft target update; one thread per parameter
__global__ void ddpg_reduce_adam_kernel(float* __restrict__ p, float* __restrict__ p_target, float* __restrict__ m,
                                        float* __restrict__ v, const float* __restrict__ slabs, int n_slabs, int n,
                                        int frozen_lo0, int frozen_hi0, int frozen_lo1, int frozen_hi1, float lr_t, DdpgHyper h,
                                        float inv_b, float* __restrict__ info_out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n && !((k >= frozen_lo0 && k < frozen_hi0) || (k >= frozen_lo1 && k < frozen_hi1))) {
        float g = 0.f;
        for (int c = 0; c < n_slabs; ++c) g += slabs[(int64_t)c * kSlab + k];
        const float mk = h.beta1 * m[k] + (1.f - h.beta1) * g;
        const float vk = h.beta2 * v[k] + (1.f - h.beta2) * g * g;
        m[k] = mk; v[k] = vk;
        const float pk = p[k] - lr_t * mk / (sqrtf(vk) + h.eps);
        p[k] = pk;
        p_target[k] = h.tau * pk + (1.f - h.tau) * p_target[k];
    }
    if (info_out && k < 2) {                                   // critic call only: loss and mean Q ride in the slab tails
        float a = 0.f;
        for (int c = 0; c < n_slabs; ++c) a += slabs[(int64_t)c * kSlab + n + k];
        info_out[k] = a * inv_b;
    }
}

// ---- the same two halves as separate steps, for learners that exchange gradients (one rank per GPU): slabs -> one
//      gradient vector (fixed order), and Adam + soft target update from a (reduced) gradient vector --------------------
__global__ void ddpg_reduce_kernel(const float* __restrict__ slabs, int n_slabs, int n, float* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    float g = 0.f;
    for (int c = 0; c < n_slabs; ++c) g += slabs[(int64_t)c * kSlab + k];
    out[k] = g;
}

__global__ void ddpg_apply_kernel(float* __restrict__ p, float* __restrict__ p_target, float* __restrict__ m, float* __restrict__ v,
                                  const float* __restrict__ grad, float grad_scale, int n, int frozen_lo0, int frozen_hi0,
                                  int frozen_lo1, int frozen_hi1, float lr_t, DdpgHyper h) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n || (k >= frozen_lo0 && k < frozen_hi0) || (k >= frozen_lo1 && k < frozen_hi1)) return;
    const float g = grad[k] * grad_scale;
    const float mk = h.beta1 * m[k] + (1.f - h.beta1) * g;
    const float vk = h.beta2 * v[k] + (1.f - h.beta2) * g * g;
    m[k] = mk; v[k] = vk;
    const float pk = p[k] - lr_t * mk / (sqrtf(vk) + h.eps);
    p[k] = pk;
    p_target[k] = h.tau * pk + (1.f - h.tau) * p_target[k];
}

// ---- minibatch rows without replacement, any size, in parallel: a keyed bijection of [0, 2^(2w)) >= count (4-round
//      Feistel network, round keys from Philox(seed; update index)) walked until it lands below count -----------------------
__global__ void replay_sample_kernel(int64_t count, int batch, PhiloxKeys keys, uint64_t update_index, int64_t* __restrict__ idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    uint32_t rk[4];
    philox4x32_10(5u << 28, (uint32_t)update_index, (uint32_t)(update_index >> 32), 0u, keys.rk, rk[0], rk[1], rk[2], rk[3]);
    int w = 1;
    while (((int64_t)1 << (2 * w)) < count) ++w;               // half width: the domain is 2^(2w) in [count, 4 count)
    const uint32_t mask = w >= 32 ? 0xFFFFFFFFu : ((1u << w) - 1u);
    uint64_t x = (uint64_t)i;
    do {
        uint32_t l = (uint32_t)(x >> w) & mask, r = (uint32_t)x & mask;
#pragma unroll
        for (int round = 0; round < 4; ++round) {
            uint32_t f = r * 0x9E3779B1u ^ rk[round];
            f ^= f >> 15; f *= 0x85EBCA77u; f ^= f >> 13; f *= 0xC2B2AE3Du; f ^= f >> 16;
            const uint32_t nl = r;
            r = (l ^ f) & mask;
            l = nl;
        }
        x = ((uint64_t)l << w) | r;
    } while ((int64_t)x >= count);                             // cycle walking keeps the map a bijection on [0, count)
    idx[i] = (int64_t)x;
}

// ---- replay ring ----------------------------------------------------------------------------------------------------
// Transition i of a vectorised env step goes to slot (head + i) mod capacity (the deque of :16-37 with the oldest
// entry dropped when full).  Observations arrive as the env's SoA rows [5][stride], actions as [n][2].
template <class T>
__global__ void replay_add_kernel(float* __restrict__ rs, float* __restrict__ ra, float* __restrict__ rr, float* __restrict__ rd,
                                  float* __restrict__ rs2, int64_t capacity, int64_t head, const T* __restrict__ obs,
                                  int64_t obs_stride, const T* __restrict__ actions, const T* __restrict__ rew,
                                  const uint8_t* __restrict__ done, const T* __restrict__ obs2, int64_t obs2_stride, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t slot = (head + i) % capacity;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        rs[slot * 5 + k] = (float)obs[k * obs_stride + i];
        rs2[slot * 5 + k] = (float)obs2[k * obs2_stride + i];
    }
    ra[slot * 2] = (float)actions[2 * i];
    ra[slot * 2 + 1] = (float)actions[2 * i + 1];
    rr[slot] = (float)rew[i];
    rd[slot] = done[i] ? 1.f : 0.f;
}

// ---- Ornstein-Uhlenbeck exploration noise (:58-78), one process per env and action dimension ----------------------------
//   x <- x + theta (mu - x) dt + sigma sqrt(dt) N(0, 1);   action += x;   envs flagged in reset_mask restart at x = 0
template <class T>
__global__ void ou_noise_kernel(double* __restrict__ x, T* __restrict__ actions, const uint8_t* __restrict__ reset_mask, int64_t n,
                                double theta, double mu, double sigma, double dt, PhiloxKeys keys, uint64_t counter, uint64_t env_base) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float z0, z1;
    ou_normals(keys, counter, env_base + (uint64_t)i, z0, z1);
    double x0 = x[2 * i], x1 = x[2 * i + 1];
    if (reset_mask && reset_mask[i]) { x0 = 0.0; x1 = 0.0; }
    const double sd = sigma * sqrt(dt);
    x0 = ou_update(x0, z0, theta, mu, sd, dt);
    x1 = ou_update(x1, z1, theta, mu, sd, dt);
    x[2 * i] = x0; x[2 * i + 1] = x1;
    actions[2 * i] = (T)((double)actions[2 * i] + x0);
    actions[2 * i + 1] = (T)((double)actions[2 * i + 1] + x1);
}

}  // namespace mr

namespace mr {
// the floats every update kernel sees: (float) of each double of mr_ddpg_hyper
static DdpgHyper to_hyper(const mr_ddpg_hyper& hp) {
    return DdpgHyper{(float)hp.gamma, (float)hp.tau, (float)hp.lr_actor, (float)hp.lr_critic, (float)hp.action_bound[0],
                     (float)hp.action_bound[1], (float)hp.adam_beta1, (float)hp.adam_beta2, (float)hp.adam_eps};
}
}  // namespace mr

extern "C" {

int32_t mr_critic_param_count(void) { return mr::kCriticParams; }

int mr_replay_add(const mr_replay* rb, int64_t head, const void* obs, int64_t obs_row_stride, const void* actions,
                  const void* rew, const uint8_t* done, const void* obs_next, int64_t obs_next_row_stride, int64_t n,
                  int32_t dtype, void* stream) {
    mr::NvtxRange nvtx_range("mr_replay_add");
    using namespace mr;
    if (!rb || !rb->s || !rb->a || !rb->r || !rb->d || !rb->s2) return fail(MR_ERR_ARG, "mr_replay_add: null replay buffer");
    if (!obs || !actions || !rew || !done || !obs_next) return fail(MR_ERR_ARG, "mr_replay_add: null argument");
    if (rb->capacity <= 0 || n < 0 || n > rb->capacity || head < 0 || head >= rb->capacity)
        return fail(MR_ERR_ARG, "mr_replay_add: need 0 <= n <= capacity and 0 <= head < capacity");
    if (n == 0) return MR_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    const int64_t st = obs_row_stride ? obs_row_stride : n, st2 = obs_next_row_stride ? obs_next_row_stride : n;
    if (dtype == MR_F64)
        replay_add_kernel<double><<<blocks, 256, 0, s>>>(rb->s, rb->a, rb->r, rb->d, rb->s2, rb->capacity, head, (const double*)obs, st,
                                                         (const double*)actions, (const double*)rew, done, (const double*)obs_next, st2, n);
    else if (dtype == MR_F32)
        replay_add_kernel<float><<<blocks, 256, 0, s>>>(rb->s, rb->a, rb->r, rb->d, rb->s2, rb->capacity, head, (const float*)obs, st,
                                                        (const float*)actions, (const float*)rew, done, (const float*)obs_next, st2, n);
    else return fail(MR_ERR_ARG, "mr_replay_add: bad dtype");
    return check_launch("mr_replay_add");
}

int mr_ou_noise_add(double* ou_state, void* actions, const uint8_t* reset_mask, int64_t n, int32_t dtype, double theta, double mu,
                    double sigma, double dt, uint64_t seed, uint64_t counter, uint64_t env_base, void* stream) {
    using namespace mr;
    if (!ou_state || !actions) return fail(MR_ERR_ARG, "mr_ou_noise_add: null argument");
    if (n < 0) return fail(MR_ERR_ARG, "mr_ou_noise_add: bad n");
    if (n == 0) return MR_OK;
    PhiloxKeys keys;
    philox_make_keys(seed, keys);
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (dtype == MR_F64) ou_noise_kernel<double><<<blocks, 256, 0, s>>>(ou_state, (double*)actions, reset_mask, n, theta, mu, sigma, dt, keys, counter, env_base);
    else if (dtype == MR_F32) ou_noise_kernel<float><<<blocks, 256, 0, s>>>(ou_state, (float*)actions, reset_mask, n, theta, mu, sigma, dt, keys, counter, env_base);
    else return fail(MR_ERR_ARG, "mr_ou_noise_add: bad dtype");
    return check_launch("mr_ou_noise_add");
}

int64_t mr_ddpg_workspace_bytes(int32_t batch) {
    if (batch <= 0) return 0;
    const int64_t tiles = (batch + mr::kTile - 1) / mr::kTile;
    const int64_t ctas = tiles < mr::kMaxCtas ? tiles : mr::kMaxCtas;
    return (int64_t)batch * 8 + ctas * mr::kSlab * 4 + 64;
}

int mr_replay_sample(int64_t count, int32_t batch, uint64_t seed, int64_t update_index, int64_t* indices_out, void* stream) {
    using namespace mr;
    if (!indices_out) return fail(MR_ERR_ARG, "mr_replay_sample: null output");
    if (batch <= 0 || count < batch) return fail(MR_ERR_ARG, "mr_replay_sample: need 0 < batch <= count");
    PhiloxKeys keys;
    philox_make_keys(seed, keys);
    replay_sample_kernel<<<(batch + 255) / 256, 256, 0, (cudaStream_t)stream>>>(count, batch, keys, (uint64_t)update_index, indices_out);
    return check_launch("mr_replay_sample");
}

int mr_ddpg_update(const mr_ddpg_state* st, const mr_replay* rb, int64_t count, int32_t batch, const int64_t* indices,
                   uint64_t seed, int64_t update_index, const mr_ddpg_hyper* hp, float* info_out, void* workspace,
                   int64_t workspace_bytes, void* stream) {
    mr::NvtxRange nvtx_range("mr_ddpg_update");
    using namespace mr;
    if (!st || !st->actor || !st->actor_target || !st->critic || !st->critic_target || !st->adam_actor_m || !st->adam_actor_v ||
        !st->adam_critic_m || !st->adam_critic_v || !st->grad_actor || !st->grad_critic)
        return fail(MR_ERR_ARG, "mr_ddpg_update: null learner state");
    if (!rb || !rb->s || !rb->a || !rb->r || !rb->d || !rb->s2) return fail(MR_ERR_ARG, "mr_ddpg_update: null replay buffer");
    if (!hp) return fail(MR_ERR_ARG, "mr_ddpg_update: null hyper-parameters");
    const bool wide = workspace != nullptr && batch > kWideBatch;              // data-parallel path for large minibatches
    if (batch <= 0 || (!wide && batch > kMaxBatch))
        return fail(MR_ERR_ARG, "mr_ddpg_update: batch must be in 1..%d (larger ones need the workspace of mr_ddpg_workspace_bytes)", kMaxBatch);
    if (count < batch || count > rb->capacity) return fail(MR_ERR_ARG, "mr_ddpg_update: need batch <= count <= capacity (the reference waits for min_batch transitions)");
    if (update_index < 1) return fail(MR_ERR_ARG, "mr_ddpg_update: update_index is Adam's step count, starting at 1");
    const DdpgHyper h = to_hyper(*hp);
    PhiloxKeys keys;
    philox_make_keys(seed, keys);
    cudaStream_t s = (cudaStream_t)stream;
    static bool attr[kMaxDevices] = {};
    const int dev = current_device();
    if (!attr[dev]) {
        cudaFuncSetAttribute(ddpg_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DdpgSmem));
        cudaFuncSetAttribute(ddpg_critic_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DdpgSmem));
        cudaFuncSetAttribute(ddpg_actor_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DdpgSmem));
        attr[dev] = true;
    }
    if (!wide) {
        ddpg_update_kernel<<<1, kDdpgThreads, sizeof(DdpgSmem), s>>>(
            st->actor, st->actor_target, st->critic, st->critic_target, st->adam_actor_m, st->adam_actor_v, st->adam_critic_m,
            st->adam_critic_v, st->grad_actor, st->grad_critic, rb->s, rb->a, rb->r, rb->d, rb->s2, count, batch, indices, keys,
            (uint64_t)update_index, h, info_out);
        return check_launch("mr_ddpg_update");
    }
    if (workspace_bytes < mr_ddpg_workspace_bytes(batch)) return fail(MR_ERR_ARG, "mr_ddpg_update: workspace too small");
    if ((uintptr_t)workspace & 15u) return fail(MR_ERR_ARG, "mr_ddpg_update: workspace must be 16-byte aligned");
    int64_t* idx = (int64_t*)workspace;
    float* slabs = (float*)((char*)workspace + (((int64_t)batch * 8 + 63) / 64) * 64);
    const int tiles = (batch + kTile - 1) / kTile;
    const int sms = sm_count(dev);
    const int ctas = tiles < sms ? tiles : (sms < kMaxCtas ? sms : kMaxCtas);
    if (indices) cudaMemcpyAsync(idx, indices, (size_t)batch * 8, cudaMemcpyDeviceToDevice, s);
    else replay_sample_kernel<<<(batch + 255) / 256, 256, 0, s>>>(count, batch, keys, (uint64_t)update_index, idx);
    const float t = (float)update_index, inv_b = 1.0f / (float)batch;
    const float corr = sqrtf(1.f - powf(h.beta2, t)) / (1.f - powf(h.beta1, t));
    ddpg_critic_grad_kernel<<<ctas, kDdpgThreads, sizeof(DdpgSmem), s>>>(st->actor_target, st->critic, st->critic_target, rb->s, rb->a,
                                                                         rb->r, rb->d, rb->s2, idx, batch, h, slabs);
    ddpg_reduce_adam_kernel<<<(kCriticParams + 255) / 256, 256, 0, s>>>(st->critic, st->critic_target, st->adam_critic_m, st->adam_critic_v,
                                                                        slabs, ctas, kCriticParams, kC_Mc, kC_T1, 0, 0,
                                                                        h.lr_critic * corr, h, inv_b, info_out);
    ddpg_actor_grad_kernel<<<ctas, kDdpgThreads, sizeof(DdpgSmem), s>>>(st->actor, st->critic, rb->s, rb->a, rb->r, rb->d, rb->s2, idx,
                                                                        batch, h, slabs);
    ddpg_reduce_adam_kernel<<<(kActorParams + 255) / 256, 256, 0, s>>>(st->actor, st->actor_target, st->adam_actor_m, st->adam_actor_v,
                                                                       slabs, ctas, kActorParams, kOffM1, kOffW2, kOffM2, kOffW3,
                                                                       h.lr_actor * corr, h, inv_b, nullptr);
    return check_launch("mr_ddpg_update");
}

int mr_ddpg_update_population(const mr_ddpg_population* pop, int64_t count, int32_t batch, int64_t update_index, float* info_out,
                              void* stream) {
    mr::NvtxRange nvtx_range("mr_ddpg_update_population");
    using namespace mr;
    const char* fn = "mr_ddpg_update_population";
    if (!pop) return fail(MR_ERR_ARG, "%s: null population", fn);
    if (pop->members < 1 || pop->members > kMaxMembers) return fail(MR_ERR_ARG, "%s: members must be in 1..%d", fn, kMaxMembers);
    const mr_ddpg_state* st = &pop->st;
    if (!st->actor || !st->actor_target || !st->critic || !st->critic_target || !st->adam_actor_m || !st->adam_actor_v ||
        !st->adam_critic_m || !st->adam_critic_v || !st->grad_actor || !st->grad_critic)
        return fail(MR_ERR_ARG, "%s: null learner state", fn);
    const mr_replay* rb = &pop->ring;
    if (!rb->s || !rb->a || !rb->r || !rb->d || !rb->s2) return fail(MR_ERR_ARG, "%s: null replay ring array", fn);
    if (!pop->hyper) return fail(MR_ERR_ARG, "%s: null hyper-parameters", fn);
    if (!pop->seeds) return fail(MR_ERR_ARG, "%s: null seeds", fn);
    if (batch <= 0 || batch > kMaxBatch) return fail(MR_ERR_ARG, "%s: batch must be in 1..%d", fn, kMaxBatch);
    if (count < batch || count > rb->capacity) return fail(MR_ERR_ARG, "%s: need batch <= count <= capacity", fn);
    if (update_index < 1) return fail(MR_ERR_ARG, "%s: update_index is Adam's step count, starting at 1", fn);
    DdpgMembers mem{};                                            // rows past `members` are not read
    for (int p = 0; p < pop->members; ++p) {
        const mr_ddpg_hyper& hp = pop->hyper[p];
        for (double v : {hp.gamma, hp.tau, hp.lr_actor, hp.lr_critic, hp.action_bound[0], hp.action_bound[1], hp.adam_beta1,
                         hp.adam_beta2, hp.adam_eps})
            if (!std::isfinite(v)) return fail(MR_ERR_ARG, "%s: hyper-parameters of member %d must be finite", fn, p);
        mem.m[p].h = to_hyper(hp);
        philox_make_keys(pop->seeds[p], mem.m[p].keys);
    }
    const DdpgStack ps{st->actor, st->actor_target, st->critic, st->critic_target, st->adam_actor_m, st->adam_actor_v,
                       st->adam_critic_m, st->adam_critic_v, st->grad_actor, st->grad_critic, rb->s, rb->a, rb->r, rb->d, rb->s2,
                       rb->capacity};
    static bool attr[kMaxDevices] = {};
    const int dev = current_device();
    if (!attr[dev]) {
        cudaFuncSetAttribute(ddpg_update_population_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DdpgSmem));
        attr[dev] = true;
    }
    ddpg_update_population_kernel<<<pop->members, kDdpgThreads, sizeof(DdpgSmem), (cudaStream_t)stream>>>(
        ps, count, batch, (uint64_t)update_index, info_out, mem);
    return check_launch(fn);
}

int mr_ddpg_gradients(const mr_ddpg_state* st, const mr_replay* rb, int64_t count, int32_t batch, const int64_t* indices,
                      uint64_t seed, int64_t update_index, const mr_ddpg_hyper* hp, int32_t which, float* grad_out,
                      void* workspace, int64_t workspace_bytes, void* stream) {
    mr::NvtxRange nvtx_range("mr_ddpg_gradients");
    using namespace mr;
    if (!st || !st->actor || !st->actor_target || !st->critic || !st->critic_target) return fail(MR_ERR_ARG, "mr_ddpg_gradients: null learner state");
    if (!rb || !rb->s || !rb->a || !rb->r || !rb->d || !rb->s2) return fail(MR_ERR_ARG, "mr_ddpg_gradients: null replay buffer");
    if (!hp || !grad_out) return fail(MR_ERR_ARG, "mr_ddpg_gradients: null argument");
    if (which != 0 && which != 1) return fail(MR_ERR_ARG, "mr_ddpg_gradients: which must be 0 (critic) or 1 (actor)");
    if (batch <= 0) return fail(MR_ERR_ARG, "mr_ddpg_gradients: bad batch");
    if (count < batch || count > rb->capacity) return fail(MR_ERR_ARG, "mr_ddpg_gradients: need batch <= count <= capacity");
    if (!workspace || workspace_bytes < mr_ddpg_workspace_bytes(batch)) return fail(MR_ERR_ARG, "mr_ddpg_gradients: workspace too small");
    if ((uintptr_t)workspace & 15u) return fail(MR_ERR_ARG, "mr_ddpg_gradients: workspace must be 16-byte aligned");
    const DdpgHyper h = to_hyper(*hp);
    PhiloxKeys keys;
    philox_make_keys(seed, keys);
    cudaStream_t s = (cudaStream_t)stream;
    static bool attr[kMaxDevices] = {};
    const int dev = current_device();
    if (!attr[dev]) {
        cudaFuncSetAttribute(ddpg_critic_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DdpgSmem));
        cudaFuncSetAttribute(ddpg_actor_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DdpgSmem));
        attr[dev] = true;
    }
    int64_t* idx = (int64_t*)workspace;
    float* slabs = (float*)((char*)workspace + (((int64_t)batch * 8 + 63) / 64) * 64);
    const int tiles = (batch + kTile - 1) / kTile;
    const int sms = sm_count(dev);
    const int ctas = tiles < sms ? tiles : (sms < kMaxCtas ? sms : kMaxCtas);
    // the same rows for the critic and the actor call of one update: given, or regenerated from (seed, update_index)
    if (indices) cudaMemcpyAsync(idx, indices, (size_t)batch * 8, cudaMemcpyDeviceToDevice, s);
    else replay_sample_kernel<<<(batch + 255) / 256, 256, 0, s>>>(count, batch, keys, (uint64_t)update_index, idx);
    if (which == 0) {
        ddpg_critic_grad_kernel<<<ctas, kDdpgThreads, sizeof(DdpgSmem), s>>>(st->actor_target, st->critic, st->critic_target, rb->s, rb->a,
                                                                             rb->r, rb->d, rb->s2, idx, batch, h, slabs);
        ddpg_reduce_kernel<<<(kCriticParams + 2 + 255) / 256, 256, 0, s>>>(slabs, ctas, kCriticParams + 2, grad_out);
    } else {
        ddpg_actor_grad_kernel<<<ctas, kDdpgThreads, sizeof(DdpgSmem), s>>>(st->actor, st->critic, rb->s, rb->a, rb->r, rb->d, rb->s2, idx,
                                                                            batch, h, slabs);
        ddpg_reduce_kernel<<<(kActorParams + 255) / 256, 256, 0, s>>>(slabs, ctas, kActorParams, grad_out);
    }
    return check_launch("mr_ddpg_gradients");
}

int mr_ddpg_apply(const mr_ddpg_state* st, int32_t which, const float* grad, double grad_scale, int64_t update_index,
                  const mr_ddpg_hyper* hp, void* stream) {
    mr::NvtxRange nvtx_range("mr_ddpg_apply");
    using namespace mr;
    if (!st || !st->actor || !st->actor_target || !st->critic || !st->critic_target || !st->adam_actor_m || !st->adam_actor_v ||
        !st->adam_critic_m || !st->adam_critic_v)
        return fail(MR_ERR_ARG, "mr_ddpg_apply: null learner state");
    if (!hp || !grad) return fail(MR_ERR_ARG, "mr_ddpg_apply: null argument");
    if (which != 0 && which != 1) return fail(MR_ERR_ARG, "mr_ddpg_apply: which must be 0 (critic) or 1 (actor)");
    if (update_index < 1) return fail(MR_ERR_ARG, "mr_ddpg_apply: update_index is Adam's step count, starting at 1");
    const DdpgHyper h = to_hyper(*hp);
    const float t = (float)update_index;
    const float corr = sqrtf(1.f - powf(h.beta2, t)) / (1.f - powf(h.beta1, t));
    cudaStream_t s = (cudaStream_t)stream;
    if (which == 0)
        ddpg_apply_kernel<<<(kCriticParams + 255) / 256, 256, 0, s>>>(st->critic, st->critic_target, st->adam_critic_m, st->adam_critic_v, grad,
                                                                      (float)grad_scale, kCriticParams, kC_Mc, kC_T1, 0, 0, h.lr_critic * corr, h);
    else
        ddpg_apply_kernel<<<(kActorParams + 255) / 256, 256, 0, s>>>(st->actor, st->actor_target, st->adam_actor_m, st->adam_actor_v, grad,
                                                                     (float)grad_scale, kActorParams, kOffM1, kOffW2, kOffM2, kOffW3,
                                                                     h.lr_actor * corr, h);
    return check_launch("mr_ddpg_apply");
}

}  // extern "C"
