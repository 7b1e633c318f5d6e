// DDPG actor forward on the 5th-generation tensor cores (tcgen05 + TMEM), fused into the rollout.
//
// The 64x64 hidden layer is 90 % of the actor's FLOPs and is GEMM-shaped once a CTA evaluates its
// 128 envs together:  D[128 envs][64] = H1[128][64] . W2[64][64].  Per env step each CTA
//   1. computes layer 1 + BN + ReLU per thread (thread = env = GEMM row) on the CUDA cores,
//   2. writes H1 to shared memory in the UMMA canonical K-major (no-swizzle) layout, split into a
//      TF32 "hi" part and the fp32 remainder "lo" (3xTF32: hi*hi + lo*hi + hi*lo keeps ~2^-21
//      relative accuracy, i.e. fp32 like the TensorFlow reference; single-pass TF32 would not meet
//      the 1e-4 bar),
//   3. one thread issues 24 tcgen05.mma (M=128, N=64, K=8, kind::tf32) accumulating into TMEM and
//      commits them to an mbarrier,
//   4. every thread reads its own row back with tcgen05.ld (TMEM lane = GEMM row = env = thread),
//      applies BN + ReLU, the 64x2 output layer, tanh and the action bound.
// W2 (hi / lo) is staged once per CTA.  No CUTLASS: descriptors are built by hand following the
// SM100 UMMA descriptor format.
#pragma once

#include <cstdint>

#include "mr_actor.cuh"

namespace mr {

constexpr int kTcRows = 128;                   // envs per CTA = UMMA M
constexpr int kTcLBO = 128;                    // bytes between the two 16-byte K chunks of one MMA
constexpr int kTcSBO = 16 * 128;               // bytes between 8-row groups (16 K-chunks of 128 B each)

struct alignas(128) ActorTcSmem {
    float a_hi[kTcRows * kActorHidden];        // 32 KB each
    float a_lo[kTcRows * kActorHidden];
    float b_hi[kActorHidden * kActorHidden];   // 16 KB each, B[n][k] = W2[k][n]
    float b_lo[kActorHidden * kActorHidden];
    float w1f[3][kActorHidden];                // layer 1 with BN folded in, rows for obs x, y, d (the goal inputs
    float b1f[kActorHidden];                   //   obs[2], obs[3] are identically 0 in this env: MR_env.py:57)
    float4 ep[kActorHidden];                   // epilogue per hidden unit: (s2, t2, w3[j][0], w3[j][1])
    float b3[2];
    alignas(8) uint64_t mbar;
    uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// byte offset of element (row, k) in the canonical K-major interleaved layout: 8x16B core matrices
__device__ __forceinline__ int tc_offset_bytes(int row, int k) {
    return (row >> 3) * kTcSBO + (k >> 2) * kTcLBO + (row & 7) * 16 + (k & 3) * 4;
}

__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t smem_addr) {
    // SM100 UMMA shared-memory descriptor: start address, leading / stride byte offsets (all >> 4),
    // version 1 at bit 46, layout type 0 (no swizzle) at bits 61-63
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(kTcLBO >> 4) << 16) | ((uint64_t)(kTcSBO >> 4) << 32) |
           ((uint64_t)1 << 46);
}

// instruction descriptor: D = F32 (1 << 4), A = B = TF32 (2 << 7, 2 << 10), K-major both, N >> 3 at 17, M >> 4 at 24
constexpr uint32_t kTcIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kActorHidden >> 3) << 17) |
                              ((uint32_t)(kTcRows >> 4) << 24);

__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(kTcIdesc), "r"(accumulate) : "memory");
}

__device__ __forceinline__ void tc_split(float v, float& hi, float& lo) {
    hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);    // the 19 bits a TF32 operand keeps
    lo = v - hi;                                               // exact; its leading bits feed the second pass
}

// the actor's parameters in shared memory: W2 hi/lo in UMMA layout, folded layer 1, epilogue constants
__device__ __forceinline__ void actor_tc_stage(ActorTcSmem& sm, const float* __restrict__ actor) {
    const int tid = threadIdx.x;
    for (int idx = tid; idx < kActorHidden * kActorHidden; idx += kTcRows) {
        const int k = idx / kActorHidden, nn = idx % kActorHidden;      // W2[k][nn] (input-major)
        float hi, lo;
        tc_split(actor[kOffW2 + idx], hi, lo);
        const int off = tc_offset_bytes(nn, k) >> 2;
        sm.b_hi[off] = hi;
        sm.b_lo[off] = lo;
    }
    if (tid < kActorHidden) {
        // tflearn inference BN  gamma * (x - mean) / sqrt(var + eps) + beta  folded to s * x + t.  Layer 1:
        // s1 multiplies the weights and bias (h = relu(b1f + sum_i obs_i * w1f_i)); layer 2: the bias joins t2
        // because the tensor core produces the bias-free product.
        const float s1 = actor[kOffG1 + tid] / sqrtf(actor[kOffV1 + tid] + kBnEps);
        const float s2 = actor[kOffG2 + tid] / sqrtf(actor[kOffV2 + tid] + kBnEps);
        sm.w1f[0][tid] = s1 * actor[kOffW1 + 0 * kActorHidden + tid];
        sm.w1f[1][tid] = s1 * actor[kOffW1 + 1 * kActorHidden + tid];
        sm.w1f[2][tid] = s1 * actor[kOffW1 + 4 * kActorHidden + tid];
        sm.b1f[tid] = s1 * (actor[kOffB1 + tid] - actor[kOffM1 + tid]) + actor[kOffBe1 + tid];
        sm.ep[tid] = make_float4(s2, actor[kOffBe2 + tid] + s2 * (actor[kOffB2 + tid] - actor[kOffM2 + tid]),
                                 actor[kOffW3 + tid * kActorOut], actor[kOffW3 + tid * kActorOut + 1]);
    }
    if (tid < 2) sm.b3[tid] = actor[kOffB3 + tid];
}

// once per CTA: parameters, TMEM allocation, mbarrier
__device__ __forceinline__ void actor_tc_setup(ActorTcSmem& sm, const float* __restrict__ actor) {
    const int tid = threadIdx.x;
    actor_tc_stage(sm, actor);
    if (tid < 32) {                                                    // one warp owns the TMEM allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(&sm.tmem_base)), "r"(64));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem_u32(&sm.mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // b_hi / b_lo visible to the tensor core
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// another actor for the CTA's next tile (population collector).  Every thread has waited for the MMAs of its last
// call, so the tensor core no longer reads the operands; the first barrier orders the epilogue's reads before the overwrite.
__device__ __forceinline__ void actor_tc_restage(ActorTcSmem& sm, const float* __restrict__ actor) {
    __syncthreads();
    actor_tc_stage(sm, actor);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

__device__ __forceinline__ void actor_tc_teardown(ActorTcSmem& sm) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(sm.tmem_base), "r"(64));
}

// One actor evaluation for the CTA's 128 envs.  `step` is the call index (mbarrier phase).
__device__ __forceinline__ void actor_tc_forward(ActorTcSmem& sm, const float obs[5], float hi0, float hi1, int step,
                                                 float act[2]) {
    const int tid = threadIdx.x;
    // ---- layer 1 (+ folded BN) + ReLU, 4 hidden units (= one 16-byte K chunk) at a time -------------
    char* a_hi = reinterpret_cast<char*>(sm.a_hi);
    char* a_lo = reinterpret_cast<char*>(sm.a_lo);
    const int row_off = (tid >> 3) * kTcSBO + (tid & 7) * 16;
    const float ox = obs[0], oy = obs[1], od = obs[4];        // obs[2] = obs[3] = 0: the goal is the origin
#pragma unroll 4
    for (int c = 0; c < kActorHidden / 4; ++c) {
        float4 acc = *reinterpret_cast<const float4*>(&sm.b1f[4 * c]);
        const float4 wx = *reinterpret_cast<const float4*>(&sm.w1f[0][4 * c]);
        const float4 wy = *reinterpret_cast<const float4*>(&sm.w1f[1][4 * c]);
        const float4 wd = *reinterpret_cast<const float4*>(&sm.w1f[2][4 * c]);
        acc.x = fmaf(od, wd.x, fmaf(oy, wy.x, fmaf(ox, wx.x, acc.x)));
        acc.y = fmaf(od, wd.y, fmaf(oy, wy.y, fmaf(ox, wx.y, acc.y)));
        acc.z = fmaf(od, wd.z, fmaf(oy, wy.z, fmaf(ox, wx.z, acc.z)));
        acc.w = fmaf(od, wd.w, fmaf(oy, wy.w, fmaf(ox, wx.w, acc.w)));
        float4 vh, vl;
        tc_split(fmaxf(acc.x, 0.f), vh.x, vl.x); tc_split(fmaxf(acc.y, 0.f), vh.y, vl.y);
        tc_split(fmaxf(acc.z, 0.f), vh.z, vl.z); tc_split(fmaxf(acc.w, 0.f), vh.w, vl.w);
        *reinterpret_cast<float4*>(a_hi + row_off + c * kTcLBO) = vh;
        *reinterpret_cast<float4*>(a_lo + row_off + c * kTcLBO) = vl;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // generic-proxy writes -> async proxy (tensor core)
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();

    // ---- layer 2 on the tensor core: 8 K-steps x (hi*hi + lo*hi + hi*lo) --------------------------
    if (tid == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d = sm.tmem_base;
        const uint32_t ah = tc_smem_u32(sm.a_hi), al = tc_smem_u32(sm.a_lo), bh = tc_smem_u32(sm.b_hi), bl = tc_smem_u32(sm.b_lo);
#pragma unroll
        for (int k = 0; k < kActorHidden / 8; ++k) {
            const uint32_t ko = k * 2 * kTcLBO;                        // 8 TF32 = two 16-byte chunks
            tc_mma(d, tc_smem_desc(ah + ko), tc_smem_desc(bh + ko), k > 0 ? 1u : 0u);
            tc_mma(d, tc_smem_desc(al + ko), tc_smem_desc(bh + ko), 1u);
            tc_mma(d, tc_smem_desc(ah + ko), tc_smem_desc(bl + ko), 1u);
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(&sm.mbar)) : "memory");
    }
    {   // wait for the MMAs of this call (bounded spin: a descriptor mistake must trap, not hang the GPU)
        const uint32_t bar = tc_smem_u32(&sm.mbar), parity = (uint32_t)step & 1u;
        uint32_t ok = 0;
        for (int spin = 0; spin < (1 << 28) && !ok; ++spin)
            asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                         : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (!ok) __trap();
    }
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- this thread's row of D: TMEM lane = env row, 64 fp32 columns ----------------------------
    uint32_t r[64];
    const uint32_t taddr = sm.tmem_base + ((uint32_t)((tid >> 5) * 32) << 16);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
        "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
        "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]),
          "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]),
          "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]),
          "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]),
          "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");

    // ---- BN + ReLU, output layer, tanh, action bound ------------------------------------------------
    float o0 = sm.b3[0], o1 = sm.b3[1];
#pragma unroll
    for (int j = 0; j < kActorHidden; ++j) {
        const float4 c = sm.ep[j];                                         // one broadcast 16-byte read per hidden unit
        const float y = fmaxf(fmaf(c.x, __uint_as_float(r[j]), c.y), 0.f);
        o0 = fmaf(y, c.z, o0); o1 = fmaf(y, c.w, o1);
    }
    act[0] = tanhf(o0) * hi0;
    act[1] = tanhf(o1) * hi1;
}

}  // namespace mr
