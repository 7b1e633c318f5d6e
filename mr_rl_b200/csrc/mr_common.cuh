// Shared device-side views and helpers of the env kernels (step / reset / rollout).
#pragma once
#include <cuda.h>            // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint, no libcuda link)
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>   // header-only: ranges cost a pointer test unless a profiler is attached

#include <cstdint>
#include <cstring>

#include "../../include/mr_rl_b200.h"
#include "mr_core.cuh"

namespace mr {

// NVTX range around an entry point's launches (nsys / ncu --nvtx group the kernels by the reference method they replace)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

int fail(int code, const char* fmt, ...);
int check_launch(const char* what);
extern int g_actor_path;  // in-rollout actor: 0 default (3xFP16 tensor cores), 1 CUDA cores, 2 3xTF32 tensor cores (mr_set_actor_path)
extern thread_local int g_step_cta_cap;   // > 0: at most this many CTAs per SM for the tiled step kernel (set around the direct host step)
extern int g_step_path;   // 0 default, 1 plain TMA, 2 vector, 3 scalar, 4 warp-specialised (mr_set_step_path)

// Per-device launch configuration cache (one process may drive several GPUs): kernel attributes are
// per device, so "done once" flags are indexed by the current device.
constexpr int kMaxDevices = 64;
inline int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev >= 0 && dev < kMaxDevices ? dev : 0;
}
// SMs of device `dev` (an index from current_device()), queried once per device
inline int sm_count(int dev) {
    static int cached[kMaxDevices] = {};
    if (!cached[dev]) {
        cudaDeviceGetAttribute(&cached[dev], cudaDevAttrMultiProcessorCount, dev);
        if (cached[dev] <= 0) cached[dev] = 148;
    }
    return cached[dev];
}

// ---- device-side views ---------------------------------------------------------------------
template <class T>
struct StateView {
    T *x, *y, *fx, *fy, *h;
    int32_t* counter;
    int32_t* cursor;
    uint8_t* status;
    double *a0, *sigma;   // optional per-env Simulator.a0 / noise_var rows (all three or none)
    uint8_t* mism;        // optional per-env Simulator.is_mismatched
};

template <class T>
struct OutView {
    T* obs;           // [5][stride]
    T* rew;
    uint8_t* done;
    T* sp;            // [2][stride]
    int64_t stride;
    bool goal;        // write the constant goal rows obs[2], obs[3] (off when the caller keeps them pre-zeroed)
    bool f32;         // T = double only: obs / rew / sp are float rows (mr_step_out.out_f32), stride counts floats
};

// one output element: the row is T, or float when the float32-output option is on (step kernels only)
template <class T>
__device__ __forceinline__ void put_out(T* row, bool f32, int64_t i, double v) {
    if constexpr (sizeof(T) == 8) { if (f32) { reinterpret_cast<float*>(row)[i] = (float)v; return; } }
    row[i] = (T)v;
}
template <class T>
__host__ __device__ __forceinline__ T* out_row(T* base, bool f32, int64_t elems) {   // base + elems in units of the row type
    if constexpr (sizeof(T) == 8) { if (f32) return reinterpret_cast<T*>(reinterpret_cast<float*>(base) + elems); }
    return base + elems;
}

struct NoiseView {
    const double* table;       // [table_len][table_stride]; local env i reads column table_col0 + i
    int64_t table_len, table_stride, table_col0;
    uint64_t seed, offset, env_base;
    const uint64_t* offset_dev;   // optional device counter added to offset (CUDA-graph replays)
};

// env-step index of this launch; read after griddepcontrol.wait (an earlier kernel of the stream may have set it)
__device__ __forceinline__ uint64_t step_offset(const NoiseView& nv) {
    return nv.offset + (nv.offset_dev ? *reinterpret_cast<const volatile uint64_t*>(nv.offset_dev) : 0ull);
}

struct TimeView { const double* t; int len; };

// 2-D TMA tensor maps of the step kernel (csrc/mr_step_tma.cuh): the SoA rows of one tensor are equally strided, so the
// rows a tile needs form a {kTile x rows} box that ONE cp.async.bulk.tensor instruction moves — the five state rows,
// obs rows (x, y) / (goal_x, goal_y), the two state_prime rows, the 16 / 24 noise-table rows of the tile.
struct StepMaps {
    CUtensorMap state;      // [5][n]      x, y, fx, fy, h          box {kTile, 5}
    CUtensorMap obs;        // [5][n]      x, y, gx, gy, d          box {kTile, 2}
    CUtensorMap sp;         // [2][n]      state_prime              box {kTile, 2}
    CUtensorMap table;      // [L][n]      noise table (fp64)       box {kTile, 16 | 24}
};
// Fills `m` for this call (maps are cached by geometry); false if the rows are not equally strided / aligned.
template <class T>
bool build_step_maps(StepMaps& m, const StateView<T>& sv, const OutView<T>& ov, const NoiseView& nv, int64_t n, int tile,
                     int table_rows);

__device__ __forceinline__ double time_at(const TimeView& tv, int c, double dt) {
    if (c < tv.len) return __ldg(tv.t + c);
    double t = __ldg(tv.t + tv.len - 1);                 // beyond the table: keep accumulating exactly
    for (int k = tv.len - 1; k < c; ++k) t += dt;
    return t;
}

// The carried step size decides how many RK45 attempts (hence noise draws) a step makes, so it
// must survive storage exactly when it equals the interval length (the common case).  fp64
// storage keeps h itself; fp32 storage keeps the ratio h / interval_length, where 1.0f is exact.
template <class T> __device__ __forceinline__ double decode_h(T raw, double il) { return (double)raw; }
template <> __device__ __forceinline__ double decode_h<float>(float raw, double il) {
    return raw == 1.0f ? il : (double)raw * il;
}
template <class T> __device__ __forceinline__ T encode_h(double h, double il) { return (T)h; }
template <> __device__ __forceinline__ float encode_h<float>(double h, double il) { return (float)(h / il); }

// 16-byte vector access helpers: VEC consecutive envs of one SoA row per thread.
template <class T, int VEC> struct Pack { T v[VEC]; };

template <class T, int VEC>
__device__ __forceinline__ Pack<T, VEC> load_pack(const T* row, int64_t i0) {
    Pack<T, VEC> p;
    if constexpr (VEC == 1) { p.v[0] = row[i0]; }
    else if constexpr (sizeof(T) * VEC == 16) {
        const int4 raw = *reinterpret_cast<const int4*>(row + i0);
        memcpy(&p, &raw, 16);
    } else if constexpr (sizeof(T) * VEC == 8) {
        const int2 raw = *reinterpret_cast<const int2*>(row + i0);
        memcpy(&p, &raw, 8);
    } else if constexpr (sizeof(T) * VEC == 4) {
        const int raw = *reinterpret_cast<const int*>(row + i0);
        memcpy(&p, &raw, 4);
    } else if constexpr (sizeof(T) * VEC == 2) {
        const short raw = *reinterpret_cast<const short*>(row + i0);
        memcpy(&p, &raw, 2);
    } else {
#pragma unroll
        for (int j = 0; j < VEC; ++j) p.v[j] = row[i0 + j];
    }
    return p;
}

template <class T, int VEC>
__device__ __forceinline__ void store_pack(T* row, int64_t i0, const Pack<T, VEC>& p) {
    if constexpr (VEC == 1) { row[i0] = p.v[0]; }
    else if constexpr (sizeof(T) * VEC == 16) {
        int4 raw; memcpy(&raw, &p, 16);
        *reinterpret_cast<int4*>(row + i0) = raw;
    } else if constexpr (sizeof(T) * VEC == 8) {
        int2 raw; memcpy(&raw, &p, 8);
        *reinterpret_cast<int2*>(row + i0) = raw;
    } else if constexpr (sizeof(T) * VEC == 4) {
        int raw; memcpy(&raw, &p, 4);
        *reinterpret_cast<int*>(row + i0) = raw;
    } else if constexpr (sizeof(T) * VEC == 2) {
        short raw; memcpy(&raw, &p, 2);
        *reinterpret_cast<short*>(row + i0) = raw;
    } else {
#pragma unroll
        for (int j = 0; j < VEC; ++j) row[i0 + j] = p.v[j];
    }
}

template <int MODE> struct NoiseOf;
template <> struct NoiseOf<MR_NOISE_NONE> { using type = NoNoise; };
template <> struct NoiseOf<MR_NOISE_TABLE> { using type = TableNoise; };
template <> struct NoiseOf<MR_NOISE_PHILOX> { using type = PhiloxNoise; };

template <int MODE>
__device__ __forceinline__ typename NoiseOf<MODE>::type make_noise(const NoiseView& nv, int64_t n, int64_t env,
                                                                   int32_t cursor, uint64_t step,
                                                                   uint32_t purpose = kPurposeNoise) {
    typename NoiseOf<MODE>::type nz;
    if constexpr (MODE == MR_NOISE_TABLE) {
        nz.col = nv.table + nv.table_col0 + env; nz.stride = nv.table_stride; nz.cursor = cursor;
        nz.len = (int32_t)nv.table_len; nz.overflow = 0;
    } else if constexpr (MODE == MR_NOISE_PHILOX) {
        nz.seek(nv.env_base + (uint64_t)env, step, purpose);
    }
    return nz;
}


// gym-style auto reset after a terminal step: the env restarts from a Philox-sampled
// init_space position (float32-rounded like gym.spaces.Box.sample, MR_env.py:172-173).
__device__ __forceinline__ void sample_init(const NoiseView& nv, int64_t i, uint64_t step, const Params& p, double& x0, double& y0) {
    double u[4];
    philox_uniform4(p, nv.env_base + (uint64_t)i, step, kPurposeInit, u);
    x0 = (double)(float)(p.init_lo[0] + (p.init_hi[0] - p.init_lo[0]) * u[0]);
    y0 = (double)(float)(p.init_lo[1] + (p.init_hi[1] - p.init_lo[1]) * u[1]);
}

// MR_Env.reset(init = (x0, y0)) in the middle of a kernel: new integrator (two RHS evaluations with action 0 and
// fresh draws), counter 0, sticky status kept.
template <int MODE, bool MISM>
__device__ __forceinline__ void auto_reset_at(Env& e, double x0, double y0, const NoiseView& nv, int64_t n, int64_t i,
                                              int32_t& cur, uint64_t step, const Params& p, int& overflow) {
    const int keep = e.status;
    auto nzr = make_noise<MODE>(nv, n, i, cur, step, kPurposeResetNoise);
    env_reset<MISM>(e, x0, y0, p.dt, p, nzr);
    e.status |= keep;
    if constexpr (MODE == MR_NOISE_TABLE) { cur = nzr.cursor; overflow |= nzr.overflow; }
}

template <int MODE, bool MISM>
__device__ __forceinline__ void auto_reset_env(Env& e, const NoiseView& nv, int64_t n, int64_t i, int32_t& cur,
                                               uint64_t step, const Params& p, int& overflow) {
    double x0, y0;
    sample_init(nv, i, step, p, x0, y0);
    auto_reset_at<MODE, MISM>(e, x0, y0, nv, n, i, cur, step, p, overflow);
}


// ---- host-side launchers, one translation unit per (storage dtype, noise mode) -----------
template <class T, int MODE>
int launch_step(const StateView<T>& sv, const T* actions, const OutView<T>& ov, const NoiseView& nv, const TimeView& tv,
                const Params& p, int64_t n, bool vec_ok, cudaStream_t s);
struct ResetRows { const double* a0; const double* sigma; const uint8_t* mism; };   // per-env MR_Env.reset arguments (or NULL)
template <class T, int MODE>
int launch_reset(const StateView<T>& sv, const T* init_xy, const uint8_t* mask, int reset_cursor, const ResetRows& rr,
                 const OutView<T>& ov, const NoiseView& nv, const Params& p, int64_t n, cudaStream_t s);

template <class T>
struct RolloutView {
    const T* actions;          // TENSOR [K][n][2] | BROADCAST [K][2]
    const float* actor;        // packed actor weights
    T* traj_xy;                // [K][2][n]
    T* traj_sp;                // [K][2][n]
    uint8_t* traj_done;        // [K][n]
    double* stats;             // [MR_STATS_LEN]
    // per-episode recording (MR_data.py:27-57): what new_iter / new_transition log, keyed on the device
    T* traj_actions;           // [K][n][2] the action applied at step k (also for in-kernel policies)
    T* traj_rew;               // [K][n]
    T* traj_reset_xy;          // [K][2][n] start position of the episode that begins after a terminal step k (auto reset)
    int32_t* traj_episode;     // [K][n] episode ordinal of env i the transition belongs to
    int32_t* traj_step;        // [K][n] step inside that episode (MR_Env.counter after the step)
    int32_t* episode_counter;  // [n] in/out: episodes env i has finished so far
    const T* reset_init;       // [reset_init_len][n][2] start positions for the auto resets (NULL: sample init_space)
    int reset_init_len;
    int k_steps;
    int action_source;
};

// The GP-corrected heading policy of the fused rollout (mr_gp_heading_policy): per env and step k the desired velocity
// vd = v_ref[k] + gain (p_ref[k] - p), then the heading search of gp_correct_heading_cheb_kernel on [lo, hi].
struct GpHeadingView {
    const double* coef_x;      // [n_coef] Chebyshev series of the two GP means on [lo, hi]
    const double* coef_y;
    const double* ref;         // [K][4] x_ref, y_ref, vx_ref, vy_ref
    double a0f, dx, dy;        // HeadingProblem
    double freq, gain;
    double lo, hi, xatol;      // search interval and tolerance, passed at run time as the standalone kernel takes them
    int n_coef, maxfun;
};

// DDPG experience collection in the fused rollout (mr_ddpg_collect): the OU process (mr_ou.cuh) and the replay ring.
struct CollectView {
    double* ou;                     // [n][2] OU state, in/out
    PhiloxKeys keys;                // of the OU seed
    double theta, mu, sd, dt;       // sd = sigma sqrt(dt), as ou_noise_kernel forms it
    uint64_t counter, env_base;     // step k draws OU sample counter + k of env env_base + i
    float *s, *a, *r, *d, *s2;      // ring rows [capacity][5] / [capacity][2] / [capacity] / [capacity] / [capacity][5]
    int64_t capacity, head;         // transition (k, i) goes to slot (head + k n + i) % capacity
    int64_t member_envs;            // population (mr_env_rollout_ddpg_collect_population): envs per member N; 0: one learner
};
// Greedy evaluation of a DDPG population (mr_ddpg_evaluate_population): env i = p N + j (N = CollectView::member_envs)
// starts episode j of member p in the launch and is frozen after its terminal step.  No state rows are read or written.
template <class T>
struct EvalView {
    const T* init;              // [N][2] start positions, or NULL: sample init_space
    double* ret;                // [n] undiscounted return, or NULL
    int32_t* length;            // [n] episode length, or NULL
    uint8_t* outcome;           // [n] 1 goal, 2 out of bounds, 3 timeout, or NULL
    uint8_t* status;            // [n] sticky MR_ENV_* flags, or NULL
    int crn;                    // common random numbers: env p N + j draws with the key of env j
};
// The fused rollout of every action source.  gh: the GP heading policy, only from mr_env_rollout_gp_heading; cv: the
// DDPG collector, only from mr_env_rollout_ddpg_collect(_population); ev (with cv->member_envs): the population
// evaluation, only from mr_ddpg_evaluate_population; all null from mr_env_rollout.
template <class T, int MODE>
int launch_rollout(const StateView<T>& sv, const RolloutView<T>& rv, const OutView<T>& ov, const NoiseView& nv,
                   const TimeView& tv, const Params& p, int64_t n, const GpHeadingView* gh, const CollectView* cv,
                   const EvalView<T>* ev, cudaStream_t s);

}  // namespace mr
