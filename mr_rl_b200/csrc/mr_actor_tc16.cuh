// DDPG actor forward (RL/MR_ddpg.py:124-149) with BOTH dense layers on the 5th-generation tensor cores, fp16 operands
// in three passes (fp32 accuracy), built so that FOUR 128-env CTAs fit an SM.
//
// Why a second tensor-core path (the TF32 one is mr_actor_tc.cuh): with 3xTF32 the A operand (hidden activations,
// hi + lo parts) takes 64 KB of shared memory per CTA and the epilogue held a 64-register TMEM row, so only two CTAs
// (8 warps) were resident per SM and nothing hid the latency of the synchronous write-H1 / MMA / read-D sequence
// (r01 ncu: 12 % warps active, issue slots 35 % busy, 0.42 eligible warps per cycle).  Here
//   * operands are fp16 pairs  v = hi + lo  (hi = fp16(v), lo = fp16(v - hi): 22 significand bits, ~2^-22 relative like
//     the 3xTF32 split) and the product is hi*hi + lo*hi + hi*lo accumulated in fp32 in TMEM: half the operand bytes
//     (A: 32 KB, W2: 16 KB), K = 16 per instruction instead of 8, twice the tensor rate;
//   * layer 1 runs on the tensor core too: A1[128 x 16] = [x, y, d, 1, 0 ...] (the goal inputs obs[2], obs[3] are
//     identically 0, MR_env.py:57), B1 = BN-folded W1 with the folded bias in the k = 3 slot; its A tile aliases the
//     first 4 KB of the layer-2 A buffers (consumed before they are written).  (Measured against layer 1 on the CUDA
//     cores with packed FFMA2 — one MMA round trip and one CTA barrier fewer, 96 FFMA2 + 64 LDS more per step:
//     1.47e10 against 1.56e10 env-steps/s, so the tensor core keeps it.);
//   * TMEM rows are read back in 16-column chunks fused with ReLU + re-split (layer 1) or BN + ReLU + the 64x2 output
//     layer (layer 2): 16 live registers instead of 64;
//   -> 53 KB shared memory, 128 TMEM columns and <= 128 registers per CTA: 4 CTAs = 16 warps per SM, so one CTA's MMA
//   round trips overlap the CUDA-core work (operand split, epilogue, the fp64 env step) of the three others.
// Range: fp16 operands overflow beyond 65504 — an observation or hidden activation that large turns the action into
// NaN, which the env flags as MR_ENV_NONFINITE (a loud failure; MR_Env's observation bounds are 5000 / 80000 and
// batch-normalised activations are O(1-10)).  The TF32 path keeps fp32 range and stays selectable (MR_ACTOR_PATH=tf32).  Descriptors are hand-built (SM100 UMMA, K-major, no swizzle), no CUTLASS.
#pragma once

#include <cuda_fp16.h>

#include <cstdint>

#include "mr_actor.cuh"

namespace mr {

constexpr int kT16Rows = 128;                  // envs per CTA = UMMA M
constexpr int kT16LBO = 128;                   // bytes between adjacent 16-byte K chunks (8 halfs) of an 8-row group
constexpr int kT16SBO2 = 8 * 128;              // layer 2: K = 64 halfs = 8 chunks per 8-row group
constexpr int kT16SBO1 = 2 * 128;              // layer 1: K = 16 halfs = 2 chunks per 8-row group
constexpr int kT16Cols = 128;                  // TMEM columns: D1 [0, 64), D2 [64, 128)

struct alignas(128) ActorTc16Smem {
    __half a_hi[kT16Rows * kActorHidden];      // 16 KB each; bytes [0, 4096) double as the layer-1 A tile [128 x 16]
    __half a_lo[kT16Rows * kActorHidden];
    __half b2_hi[kActorHidden * kActorHidden]; // 8 KB each, B2[n][k] = W2[k][n]
    __half b2_lo[kActorHidden * kActorHidden];
    __half b1_hi[kActorHidden * 16];           // 2 KB each, B1[n][k]: k = 0, 1, 2 folded W1 rows of x, y, d; k = 3 folded bias
    __half b1_lo[kActorHidden * 16];
    float4 ep[kActorHidden];                   // epilogue per PAIR of hidden units (j, j+1): ep[j] = (s2_j, s2_j+1, t2_j, t2_j+1),
                                               //   ep[j+1] = (w3[j][0], w3[j+1][0], w3[j][1], w3[j+1][1])
    float b3[2];
    alignas(8) uint64_t mbar[2];               // completion of the layer-1 / layer-2 MMAs
    uint64_t desc[8];                          // UMMA descriptors of the operand tiles (loop-invariant: built once, the
                                               //   issuing thread only adds the K offset): A1 hi/lo, B1 hi/lo, A2 hi/lo, B2 hi/lo
    uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t t16_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// byte offset of element (row, k) in the canonical K-major layout of 16-bit operands: 8 x 16 B core matrices
__device__ __forceinline__ int t16_offset_bytes(int row, int k, int sbo) {
    return (row >> 3) * sbo + (k >> 3) * kT16LBO + (row & 7) * 16 + (k & 7) * 2;
}

__device__ __forceinline__ uint64_t t16_desc(uint32_t smem_addr, int sbo) {
    // SM100 UMMA shared-memory descriptor: start address, leading / stride byte offsets (all >> 4), version 1 at
    // bit 46, layout type 0 (no swizzle) at bits 61-63
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(kT16LBO >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
           ((uint64_t)1 << 46);
}

// instruction descriptor: D = F32 (1 << 4), A = B = F16 (0 at bits 7, 10), K-major both, N >> 3 at 17, M >> 4 at 24
constexpr uint32_t kT16Idesc = (1u << 4) | ((uint32_t)(kActorHidden >> 3) << 17) | ((uint32_t)(kT16Rows >> 4) << 24);

__device__ __forceinline__ void t16_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(kT16Idesc), "r"(accumulate) : "memory");
}

// Blackwell packed fp32 arithmetic (FFMA2 / FADD2 in SASS): two independent fp32 operations per instruction
__device__ __forceinline__ float2 t16_fma2(float2 a, float2 b, float2 c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d)
        : "l"(*reinterpret_cast<const uint64_t*>(&a)), "l"(*reinterpret_cast<const uint64_t*>(&b)), "l"(*reinterpret_cast<const uint64_t*>(&c)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 t16_sub2(float2 a, float2 b) {
    uint64_t d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<const uint64_t*>(&a)), "l"(*reinterpret_cast<const uint64_t*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}

// (a, b) -> packed fp16 pairs hi and lo with a = hi.x + lo.x, b = hi.y + lo.y to ~2^-22 relative
__device__ __forceinline__ void t16_split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 back = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - back.x, b - back.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// ReLU fused into the split (hidden activations): hi = fp16(max(v, 0)) rounded TOWARDS ZERO, so the remainder is never
// negative and the lo conversion may apply ReLU too — which also zeroes the lanes where v < 0 (hi = 0, remainder = v).
// One cvt.relu instead of two FMNMX + cvt per pair; 11 + 11 significand bits, 2^-21 relative like 3xTF32.
__device__ __forceinline__ void t16_split2_relu(float a, float b, uint32_t& hi, uint32_t& lo) {
    asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));       // d = {hi half: first source, lo half: second}
    const float2 rem = t16_sub2(make_float2(a, b), __half22float2(*reinterpret_cast<const __half2*>(&hi)));
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(rem.y), "f"(rem.x));
}

// tanh to ~1e-6 relative from one ex2 and one rcp (tanhf's polynomial + exp path is ~25 instructions; the 1e-4 bar on
// the actions does not need it): tanh x = sign(x) (1 - 2 / (exp(2|x|) + 1)), and x (1 - x^2/3) where that cancels
__device__ __forceinline__ float t16_tanh(float x) {
    const float ax = fabsf(x);
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(ax * 2.8853900817779268f));   // exp(2|x|)
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    const float big = fmaf(-2.0f, r, 1.0f);
    const float small = ax * fmaf(ax * ax, -0.3333333333f, 1.0f);
    return copysignf(ax < 0.02f ? small : big, x);
}

__device__ __forceinline__ void t16_wait(uint64_t* mbar, uint32_t parity) {
    // try_wait suspends the thread in hardware until the phase completes or the hinted time passes, so the loop body
    // normally runs once or twice (the first version polled from C: 14 polls of 6 instructions per wait, 9 % of the
    // kernel's issue slots).  Bounded: a descriptor mistake must trap, not hang the GPU.
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        ".reg .u32 c;\n"
        "mov.u32 c, 0;\n"
        "T16_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, 0x4000;\n"
        "@p bra T16_DONE_%=;\n"
        "add.u32 c, c, 1;\n"
        "setp.lt.u32 q, c, 0x4000000;\n"
        "@q bra T16_WAIT_%=;\n"
        "trap;\n"
        "T16_DONE_%=:\n"
        "}\n" ::"r"(t16_smem_u32(mbar)), "r"(parity) : "memory");
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void t16_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// weights split into fp16 hi / lo in UMMA layout, folded BN constants
__device__ __forceinline__ void actor_tc16_stage(ActorTc16Smem& sm, const float* __restrict__ actor) {
    const int tid = threadIdx.x;
    char* b2h = reinterpret_cast<char*>(sm.b2_hi);
    char* b2l = reinterpret_cast<char*>(sm.b2_lo);
    for (int idx = tid; idx < kActorHidden * kActorHidden; idx += kT16Rows) {
        const int k = idx / kActorHidden, nn = idx % kActorHidden;      // W2[k][nn] (input-major)
        const float w = actor[kOffW2 + idx];
        const __half h = __float2half_rn(w);
        const int off = t16_offset_bytes(nn, k, kT16SBO2);
        *reinterpret_cast<__half*>(b2h + off) = h;
        *reinterpret_cast<__half*>(b2l + off) = __float2half_rn(w - __half2float(h));
    }
    char* b1h = reinterpret_cast<char*>(sm.b1_hi);
    char* b1l = reinterpret_cast<char*>(sm.b1_lo);
    for (int idx = tid; idx < kActorHidden * 16; idx += kT16Rows) {
        const int nn = idx >> 4, k = idx & 15;
        // tflearn inference BN  gamma * (x - mean) / sqrt(var + eps) + beta  folded to s * x + t: s1 multiplies the
        // layer-1 weights, the folded bias rides in the k = 3 column against the constant 1 of the A tile
        const float s1 = actor[kOffG1 + nn] / sqrtf(actor[kOffV1 + nn] + kBnEps);
        float w = 0.f;
        if (k == 0) w = s1 * actor[kOffW1 + 0 * kActorHidden + nn];
        else if (k == 1) w = s1 * actor[kOffW1 + 1 * kActorHidden + nn];
        else if (k == 2) w = s1 * actor[kOffW1 + 4 * kActorHidden + nn];
        else if (k == 3) w = s1 * (actor[kOffB1 + nn] - actor[kOffM1 + nn]) + actor[kOffBe1 + nn];
        const __half h = __float2half_rn(w);
        const int off = t16_offset_bytes(nn, k, kT16SBO1);
        *reinterpret_cast<__half*>(b1h + off) = h;
        *reinterpret_cast<__half*>(b1l + off) = __float2half_rn(w - __half2float(h));
    }
    if (tid < kActorHidden) {
        // layer 2: the bias joins t2 because the tensor core produces the bias-free product
        const float s2 = actor[kOffG2 + tid] / sqrtf(actor[kOffV2 + tid] + kBnEps);
        const float t2 = actor[kOffBe2 + tid] + s2 * (actor[kOffB2 + tid] - actor[kOffM2 + tid]);
        float* e = reinterpret_cast<float*>(sm.ep) + (tid >> 1) * 8 + (tid & 1);   // slot of this unit inside its pair
        e[0] = s2; e[2] = t2; e[4] = actor[kOffW3 + tid * kActorOut]; e[6] = actor[kOffW3 + tid * kActorOut + 1];
    }
    if (tid < 2) sm.b3[tid] = actor[kOffB3 + tid];
}

// once per CTA: the weights, TMEM allocation, mbarriers
__device__ __forceinline__ void actor_tc16_setup(ActorTc16Smem& sm, const float* __restrict__ actor) {
    const int tid = threadIdx.x;
    actor_tc16_stage(sm, actor);
    if (tid < 32) {                                                    // one warp owns the TMEM allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(t16_smem_u32(&sm.tmem_base)), "r"(kT16Cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        sm.desc[0] = t16_desc(t16_smem_u32(sm.a_hi), kT16SBO1); sm.desc[1] = t16_desc(t16_smem_u32(sm.a_lo), kT16SBO1);
        sm.desc[2] = t16_desc(t16_smem_u32(sm.b1_hi), kT16SBO1); sm.desc[3] = t16_desc(t16_smem_u32(sm.b1_lo), kT16SBO1);
        sm.desc[4] = t16_desc(t16_smem_u32(sm.a_hi), kT16SBO2); sm.desc[5] = t16_desc(t16_smem_u32(sm.a_lo), kT16SBO2);
        sm.desc[6] = t16_desc(t16_smem_u32(sm.b2_hi), kT16SBO2); sm.desc[7] = t16_desc(t16_smem_u32(sm.b2_lo), kT16SBO2);
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(t16_smem_u32(&sm.mbar[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(t16_smem_u32(&sm.mbar[1])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // weights visible to the tensor core
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// another actor for the persistent CTA's next tile (population collector).  Every thread has waited for the MMAs of its
// last call, so the tensor core no longer reads the operands; the first barrier orders the epilogue's reads before the
// overwrite.  TMEM, mbarriers and descriptors stay.
__device__ __forceinline__ void actor_tc16_restage(ActorTc16Smem& sm, const float* __restrict__ actor) {
    __syncthreads();
    actor_tc16_stage(sm, actor);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

__device__ __forceinline__ void actor_tc16_teardown(ActorTc16Smem& sm) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(sm.tmem_base), "r"(kT16Cols));
}

// One actor evaluation for the CTA's 128 envs (thread = env = GEMM row = TMEM lane).  `step` = call index (mbarrier phase).
// fill1 / fill2: work of the caller that does not depend on the action, run by every thread between the issue of the
// layer-1 / layer-2 MMAs and the wait for them (the rollout draws the env step's process noise there), so the MMA round
// trips are covered by the warp's own instructions and not only by the other CTAs of the SM.
struct T16NoFill { __device__ __forceinline__ void operator()() const {} };
template <class F1 = T16NoFill, class F2 = T16NoFill>
__device__ __forceinline__ void actor_tc16_forward(ActorTc16Smem& sm, const float obs[5], float hi0, float hi1, int step,
                                                   float act[2], F1 fill1 = F1(), F2 fill2 = F2()) {
    const int tid = threadIdx.x;
    const uint32_t parity = (uint32_t)step & 1u;
    char* a_hi = reinterpret_cast<char*>(sm.a_hi);
    char* a_lo = reinterpret_cast<char*>(sm.a_lo);
    const uint32_t lane_addr = sm.tmem_base + ((uint32_t)((tid >> 5) * 32) << 16);

    // ---- layer-1 A tile: [x, y, d, 1, 0, 0, 0, 0 | 0 x 8] as fp16 hi / lo -----------------------------------
    {
        uint32_t h0, l0, h1, l1;
        t16_split2(obs[0], obs[1], h0, l0);
        t16_split2(obs[4], 1.0f, h1, l1);
        const int off = (tid >> 3) * kT16SBO1 + (tid & 7) * 16;
        *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(h0, h1, 0u, 0u);
        *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(l0, l1, 0u, 0u);
        *reinterpret_cast<uint4*>(a_hi + off + kT16LBO) = make_uint4(0u, 0u, 0u, 0u);
        *reinterpret_cast<uint4*>(a_lo + off + kT16LBO) = make_uint4(0u, 0u, 0u, 0u);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // generic-proxy writes -> async proxy (tensor core)
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d1 = sm.tmem_base;
        const uint64_t ah = sm.desc[0], al = sm.desc[1], bh = sm.desc[2], bl = sm.desc[3];
        t16_mma(d1, ah, bh, 0u);
        t16_mma(d1, al, bh, 1u);
        t16_mma(d1, ah, bl, 1u);
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(t16_smem_u32(&sm.mbar[0])) : "memory");
    }
    fill1();
    t16_wait(&sm.mbar[0], parity);

    // ---- H1 = relu(D1) re-split into the layer-2 A operand, 16 hidden units at a time -----------------------------
    {
        const int row_off = (tid >> 3) * kT16SBO2 + (tid & 7) * 16;
#pragma unroll
        for (int q = 0; q < kActorHidden / 16; ++q) {
            uint32_t r[16];
            t16_ld16(lane_addr + q * 16, r);
            uint32_t h[8], l[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
                t16_split2_relu(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]), h[j], l[j]);
            *reinterpret_cast<uint4*>(a_hi + row_off + (2 * q) * kT16LBO) = make_uint4(h[0], h[1], h[2], h[3]);
            *reinterpret_cast<uint4*>(a_hi + row_off + (2 * q + 1) * kT16LBO) = make_uint4(h[4], h[5], h[6], h[7]);
            *reinterpret_cast<uint4*>(a_lo + row_off + (2 * q) * kT16LBO) = make_uint4(l[0], l[1], l[2], l[3]);
            *reinterpret_cast<uint4*>(a_lo + row_off + (2 * q + 1) * kT16LBO) = make_uint4(l[4], l[5], l[6], l[7]);
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d2 = sm.tmem_base + kActorHidden;
        const uint64_t ah = sm.desc[4], al = sm.desc[5], bh = sm.desc[6], bl = sm.desc[7];
#pragma unroll
        for (int k = 0; k < kActorHidden / 16; ++k) {
            const uint64_t ko = (uint64_t)((k * 2 * kT16LBO) >> 4);    // 16 halfs = two 16-byte chunks, in the address field's units
            t16_mma(d2, ah + ko, bh + ko, k > 0 ? 1u : 0u);
            t16_mma(d2, al + ko, bh + ko, 1u);
            t16_mma(d2, ah + ko, bl + ko, 1u);
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(t16_smem_u32(&sm.mbar[1])) : "memory");
    }
    fill2();
    t16_wait(&sm.mbar[1], parity);

    // ---- BN + ReLU, 64 x 2 output layer, tanh, action bound ---------------------------------------------------------
    float2 o0 = make_float2(sm.b3[0], 0.f), o1 = make_float2(sm.b3[1], 0.f);   // (even units, odd units) partial sums
#pragma unroll
    for (int q = 0; q < kActorHidden / 16; ++q) {
        uint32_t r[16];
        t16_ld16(lane_addr + kActorHidden + q * 16, r);
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
            const float4 bn = sm.ep[q * 16 + j], w3 = sm.ep[q * 16 + j + 1];   // two broadcast 16-byte reads per pair of units
            float2 y = t16_fma2(make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), make_float2(bn.x, bn.y),
                                make_float2(bn.z, bn.w));
            y.x = fmaxf(y.x, 0.f); y.y = fmaxf(y.y, 0.f);
            o0 = t16_fma2(y, make_float2(w3.x, w3.y), o0);
            o1 = t16_fma2(y, make_float2(w3.z, w3.w), o1);
        }
    }
    act[0] = t16_tanh(o0.x + o0.y) * hi0;
    act[1] = t16_tanh(o1.x + o1.y) * hi1;
}

}  // namespace mr
