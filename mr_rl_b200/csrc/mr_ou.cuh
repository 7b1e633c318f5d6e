// One step of the Ornstein-Uhlenbeck exploration noise (RL/MR_ddpg.py:58-78), shared by ou_noise_kernel (mr_ddpg.cu) and
// the collecting actor source of the fused rollout (mr_rollout.inl), so that both advance the process with the same
// instructions and the fused collector stays bit-identical to mr_ou_noise_add.
#pragma once
#include "mr_core.cuh"

namespace mr {

// the two standard normals of OU sample `counter` of env `env`: the fp32 Box-Muller pair of Philox4x32-10, purpose 3 << 28
__device__ __forceinline__ void ou_normals(const PhiloxKeys& keys, uint64_t counter, uint64_t env, float& z0, float& z1) {
    uint32_t o0, o1, o2, o3;
    philox4x32_10(3u << 28, (uint32_t)counter, (uint32_t)env, ((uint32_t)(env >> 32) & 0xFFFFu) | ((uint32_t)(counter >> 32) << 16),
                  keys.rk, o0, o1, o2, o3);
    box_muller(o0, o1, z0, z1);
}

// x + theta (mu - x) dt + sd z, sd = sigma sqrt(dt): the next value of one action dimension's process
__device__ __forceinline__ double ou_update(double x, float z, double theta, double mu, double sd, double dt) {
    return x + theta * (mu - x) * dt + sd * (double)z;
}

}  // namespace mr
