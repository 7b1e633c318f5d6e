// Single-step kernel, Blackwell form: a persistent CTA streams tiles of 128 (fp64 storage) / 256 (fp32) envs through
// shared memory with TMA copies in BOTH directions — 2-D tensor-map boxes (cp.async.bulk.tensor.2d) for the equally
// strided rows of one tensor, 1-D bulk copies (cp.async.bulk) for single rows — completed through mbarriers (loads)
// and bulk groups (stores).
//
//   HBM --TMA--> smem in[stage]  --LDS--> registers (one env per thread) --STS--> smem out[stage] --TMA--> HBM
//
// Loads of tile k+1..k+2 are in flight while tile k is integrated and the stores of tile k-1
// drain, so the bytes in flight per SM no longer depend on occupancy or on how many registers
// the fp64 RK45 controller needs.  Rows are SoA, so every copy moves contiguous 1-4 KB lines; the goal rows (always 0,
// MR_env.py:57) are stored from one shared zero line.  One elected thread issues all copies; the tile costs one CTA
// barrier (generated noise, fp32 noise-free) or two (fp64 noise-free, table noise) — see OneBarrier below.
#pragma once

#include "mr_common.cuh"

namespace mr {

// input stages in flight per CTA.  Measured with the tensor-map copies (2^20 envs, fp64, sigma 0 / 1): 2 stages 30.3 / 29.4 us,
// 3 stages 27.7 / 29.6 us, 4 stages 28.7 / 29.9 us.
#ifndef MR_STAGES_IN
#define MR_STAGES_IN 3
#endif
// envs per tile == threads per CTA.  Measured on B200 (2^20 envs): fp64 128 -> 30.9 us, 256 -> 32.2 us;
// fp32 128 -> 27.6 us, 256 -> 25.6 us.  Later, with generated noise (sigma 0 / 1, fp64): 128 -> 29.1 / 32.8 us,
// 64 -> 28.8 / 35.6 us, 32 (one warp per CTA, no CTA barrier needed) -> 30.8 / 36.3 us; and issuing the loads from
// warp 0 and the stores from warp 1 (to halve the issuing warp's extra work): 28.6 / 33.8 us — no gain.  Re-measured with
// one barrier per tile (sigma 0 / 1, fp64): 128 -> 27.9 / 28.6 us, 256 -> 28.9 / 28.6 us, 64 -> 29.6 / 31.2 us.
// Also measured: replacing the two CTA barriers per tile by mbarrier hand-offs (consumers arrive on "inputs read" /
// "outputs written" barriers that only the issuing thread waits on, plus an "output stage free" barrier for the
// consumers), so warps never wait for each other: 36.1 / 40.9 us with 128 arrivals, 37.0 / 41.5 us with one arrival
// per warp — the barriers are the cheaper mechanism here.  Round 2 repeated it on top of the tensor-map copies with a
// ROTATING issuer (warp it % 4 issues tile it's copies, so no warp is permanently ~100 instructions behind) and one
// mbarrier arrival per warp: bit-identical results, 37.2 / 35.6 us against 28.0 / 29.6 us — same verdict.
#ifdef MR_TILE
template <class T> struct TileOf { static constexpr int value = MR_TILE; };
#else
template <class T> struct TileOf { static constexpr int value = sizeof(T) == 8 ? 128 : 256; };
#endif
constexpr int kStagesIn = MR_STAGES_IN;
constexpr int kStagesOut = 2;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait suspends the warp in hardware until the phase completes or a time limit passes (it is not a poll), so the
// loop normally runs once.  MR_MBAR_SUSPEND_NS > 0 passes an explicit suspend-time hint.
#ifndef MR_MBAR_SUSPEND_NS
#define MR_MBAR_SUSPEND_NS 0
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
#if MR_MBAR_SUSPEND_NS > 0
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity), "r"((uint32_t)MR_MBAR_SUSPEND_NS) : "memory");
#else
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
#endif
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_store(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
// 2-D tensor-map forms (UTMALDG / UTMASTG): one instruction moves a {box_cols x box_rows} box of a strided 2-D tensor
__device__ __forceinline__ void tensor_load_2d(void* smem_dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tensor_store_2d(const CUtensorMap* map, int32_t c0, int32_t c1, const void* smem_src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(smem_src)) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <class T, int kTile>
struct alignas(128) TileIn {
    T x[kTile], y[kTile], fx[kTile], fy[kTile], h[kTile];
    T act[2 * kTile];
    int32_t counter[kTile];
};

template <class T, int kTile>
struct alignas(128) TileOut {
    T x[kTile], y[kTile], fx[kTile], fy[kTile], h[kTile];
    T d[kTile], rew[kTile], spx[kTile], spy[kTile];
    int32_t counter[kTile];
    uint8_t done[kTile];
};

// Table-noise (parity) mode: the draws an env consumes in one step are table rows cursor .. cursor+15 (+23 when
// mismatched: 3 draws per RHS evaluation, MR_simulator.py:78-80) of its column.  Envs of a tile normally share the
// cursor (every step of the common regime takes 16 draws), so those rows of the tile are kNoiseRows contiguous
// kTile*8-byte lines of the [L][n] table: they are bulk-copied with the state rows.  An env whose cursor is elsewhere
// (more RK45 attempts, an auto reset) reads the table from global memory for the rows the stage does not hold.
template <int MODE, bool MISM> struct NoiseRows { static constexpr int value = 0; };
template <bool MISM> struct NoiseRows<MR_NOISE_TABLE, MISM> { static constexpr int value = MISM ? 24 : 16; };
// input stages: the noise rows are read during the integration, so their stage is re-filled only after the tile is
// done (2 stages: one being consumed, one in flight); the other modes copy their inputs to registers first (3 stages)
template <int MODE> struct StagesIn { static constexpr int value = MODE == MR_NOISE_TABLE ? 2 : kStagesIn; };
// ONE CTA barrier per tile instead of two where it pays.  Barrier [A] ("inputs copied to registers, output stage free")
// exists only because the refill of in[s] and the re-use of out[so] are decided right after it; with a third output
// stage and the refill issued after barrier [B] both hand-offs ride on [B]: the issuing thread waits (after committing
// tile it's stores) until the stores of tile it-1 have left shared memory, which frees the stage tile it+2 writes — and
// every thread passes [B] of tile it+1 before it gets there.  The refill then starts one compute phase later (two tiles
// in flight instead of three), which only the memory-bound case feels.  Measured (B200, 2^20 envs, us per launch, two
// barriers -> one): generated noise fp64 29.6 -> 28.6, fp32 26.5 -> 26.3; noise-free fp32 22.8 -> 22.2, but noise-free
// fp64 27.9 -> 30.4 (a fourth input stage does not fit beside the third output stage at 4 CTAs per SM), so that case
// keeps two barriers; the table mode is bounded by its noise stages and keeps them too.  -DMR_ONE_BARRIER=0: never.
#ifndef MR_ONE_BARRIER
#define MR_ONE_BARRIER 1
#endif
template <class T, int MODE> struct OneBarrier {
    static constexpr bool value = MR_ONE_BARRIER && (MODE == MR_NOISE_PHILOX || (MODE == MR_NOISE_NONE && sizeof(T) == 4));
};
template <class T, int MODE> struct StagesOut { static constexpr int value = OneBarrier<T, MODE>::value ? 3 : kStagesOut; };

template <int kTile, int ROWS>
struct alignas(128) TileNoiseIn {
    double z[ROWS][kTile];
    int32_t cursor[kTile];
    int32_t base, rows;                 // the stage holds table rows [base, base + rows) of the tile's columns
};
template <int kTile> struct TileNoiseIn<kTile, 0> {};
template <int kTile, int ROWS> struct alignas(128) TileNoiseOut { int32_t cursor[kTile]; };
template <int kTile> struct TileNoiseOut<kTile, 0> {};

struct TileTableNoise {                 // TableNoise with the common rows served from shared memory
    static constexpr bool kActive = true;
    static constexpr bool kCompress = false;
    const double* stage;                // &z[0][tid] of the tile's stage, row stride = stage_stride
    const double* col;                  // &table[0][env]
    int64_t stride;
    int32_t stage_stride, base, rows;
    int32_t cursor, len;
    int overflow;
    template <class P> __device__ __forceinline__ double next(const P&) {
        double z = 0.0;
        const uint32_t k = (uint32_t)(cursor - base);
        if (k < (uint32_t)rows) z = stage[k * stage_stride];
        else if (cursor < len) z = col[(int64_t)cursor * stride];
        else overflow = 1;
        ++cursor;
        return z;
    }
};

// MR_RNG_PREFETCH = 1 (measured and rejected, kept as a build option): the generated-noise kernel draws the NEXT tile's
// eight normals per env while it integrates the current tile and parks them in shared memory (each thread reads back its
// own values, no barrier involved), which takes the draws out of the dependency chain "draw -> attempt" and leaves them
// to the scheduler.  B200, 2^20 envs: fp64 storage 31.7 us against 30.9 us without it, fp32 storage 27.9 against 28.2 us
// — the kernel is short of issue slots per resident warp, not of independent work inside a warp.
#ifndef MR_RNG_PREFETCH
#define MR_RNG_PREFETCH 0
#endif

template <class T, int MODE = MR_NOISE_NONE, bool MISM = false, int kTile = TileOf<T>::value>
struct StepSmem {
    static constexpr int kIn = StagesIn<MODE>::value;
    TileIn<T, kTile> in[kIn];
    static constexpr int kOut = StagesOut<T, MODE>::value;
    TileOut<T, kTile> out[kOut];
    TileNoiseIn<kTile, NoiseRows<MODE, MISM>::value> nin[kIn];
    TileNoiseOut<kTile, NoiseRows<MODE, MISM>::value> nout[kOut];
    alignas(128) T zero[2 * kTile];         // the two goal rows as one {kTile x 2} box
    alignas(16) float4 zpre[(MR_RNG_PREFETCH && MODE == MR_NOISE_PHILOX && !MISM) ? 2 * kTile : 1];   // next tile's normals
    alignas(8) uint64_t full[kIn];
};

// at least 16 warps per SM (<= 128 registers): the generated-noise variant would otherwise take 136.
// Measured at 2^20 envs (sigma 0 / 1): fp64 storage 16 warps 29.1 / 32.6 us, 20 warps 30.0 / 35.4, 24 warps 30.5 / 35.3
// (the spills cost more than the occupancy gives); fp32 storage 16 warps 27.4 / 32.3 us, 24 warps 23.9 / 29.7 us
// (half the bytes per env: latency hiding matters more) -> 24 warps for the 256-env fp32 tile.
#ifndef MR_TMA_WARPS
#define MR_TMA_WARPS 16
#endif
#ifndef MR_TMA_WARPS_F32
#define MR_TMA_WARPS_F32 24
#endif
template <class T> struct TmaWarps { static constexpr int value = sizeof(T) == 4 ? MR_TMA_WARPS_F32 : MR_TMA_WARPS; };
// resident CTAs per SM the launch bound asks for: the table mode is limited by its shared-memory stages instead
template <class T, int MODE> struct TmaMinCtas {
    static constexpr int value = MODE == MR_NOISE_TABLE ? 1 : TmaWarps<T>::value * 32 / TileOf<T>::value;
};

// TMAP: the equally strided rows of one tensor move as 2-D tensor-map boxes (one instruction for the five state rows, the
// obs (x, y) pair, the goal pair, the state_prime pair, the tile's 16 / 24 noise-table rows) instead of one 1-D bulk copy
// per row: 8-9 copy instructions per tile instead of 19-20 (table mode 10 instead of 36), all issued by one thread that
// also integrates an env, i.e. by the warp every other warp of the CTA waits for at the tile's two barriers.
// STD: the launch has the standard outputs — actions and output rows in the storage type, obs with its goal rows, rew and
// done, no state_prime, auto reset on — so the per-tile tests of those options fold away at compile time (tensor maps only).
template <class T, int MODE, bool MISM, bool TMAP, bool STD = false>
__global__ void __launch_bounds__(TileOf<T>::value, TmaMinCtas<T, MODE>::value)
env_step_tma_kernel(StateView<T> st, const T* __restrict__ actions, OutView<T> out, NoiseView nv, TimeView tv,
                    Params p, int64_t n_tiles, int64_t n_total, const __grid_constant__ StepMaps maps) {
    static_assert(!STD || TMAP, "the standard-output form moves its rows with tensor maps");
    constexpr int kTile = TileOf<T>::value;
    constexpr int kSI = StagesIn<MODE>::value;
    constexpr int kNR = NoiseRows<MODE, MISM>::value;
    constexpr bool kTable = MODE == MR_NOISE_TABLE;
    constexpr bool kOneBar = OneBarrier<T, MODE>::value;
    constexpr int kSO = StagesOut<T, MODE>::value;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using Smem = StepSmem<T, MODE, MISM>;
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x;
    const int64_t first = blockIdx.x, stride = gridDim.x;

    if (tid == 0) {
        for (int s = 0; s < kSI; ++s) mbar_init(&sm.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    sm.zero[tid] = (T)0; sm.zero[kTile + tid] = (T)0;   // kTile threads
    fence_async_smem();
    __syncthreads();
    // Programmatic dependent launch: everything above (smem carve-up, mbarrier init) overlaps the tail of
    // the previous launch in the stream; the state rows it wrote are only touched after this wait.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");

    constexpr uint32_t kRow = kTile * sizeof(T);
    const bool act32 = !STD && sizeof(T) == 8 && p.act_f32;  // float32 actions with fp64 storage (mr_sim_params.action_f32)
    const bool out32 = !STD && sizeof(T) == 8 && out.f32;    // float32 output rows with fp64 storage (mr_step_out.out_f32)
    const bool w_obs = STD || out.obs, w_goal = STD || out.goal, w_rew = STD || out.rew, w_done = STD || out.done;
    const bool w_sp = !STD && out.sp;
    const bool auto_reset = STD || p.auto_reset;
    const uint32_t act_bytes = act32 ? kTile * 8u : 2u * kRow;
    const uint32_t kInBytes = 5 * kRow + act_bytes + kTile * 4;
    const uint64_t off = step_offset(nv);                   // env-step index of this launch (after griddepcontrol.wait)

    // Tried and rejected (measured, 2^20 envs fp64): a dedicated producer warp with mbarrier-only
    // hand-offs (no CTA barrier) — the extra warp costs a resident CTA at ~120 registers/thread:
    // sigma=1 49.5 us vs 38.5 us for this version.
    // Bulk copies are issued by ONE elected thread.  Measured on B200 (2^20 envs, fp64, sigma=0):
    // 1 issuing thread 32.2 us, elected lanes of 2 / 8 warps 36.0 / 36.2 us, 15 lanes of warp 0
    // 53 us (cp.async.bulk takes uniform operands, divergent issue serialises through R2UR).
#ifndef MR_ISSUE_WARPS
#define MR_ISSUE_WARPS 1
#endif
    constexpr int kWarps = MR_ISSUE_WARPS;                  // 1: a single issuing thread
    const int warp = tid >> 5;
    const bool elect = (tid & 31) == 0 && warp < kWarps;
    // Copy plumbing hoisted out of the tile loop: a CTA's tiles start kTile * gridDim.x envs apart and n < 2^31, so the
    // loop advances one unsigned 32-bit env index (a few tiles past the end it still compares correctly) that is also the
    // TMA coordinate, and every row address is a base fixed before the loop plus that index.
    const uint32_t env_stride = (uint32_t)stride * kTile;
    const uint32_t n_full = (uint32_t)(n_tiles * kTile);   // envs covered by whole tiles
    const char* const act_base = (const char*)actions;
    const uint32_t act_el = act32 ? 8u : 2u * (uint32_t)sizeof(T);   // action bytes per env
    int32_t* const ctr_row = st.counter;
    T* const d_row = w_obs ? out.obs + 4 * out.stride : nullptr;
    // cbase (table mode): the noise cursor of the tile's first env = first table row to stage
    auto issue_loads = [&](int s, uint32_t i0, int32_t cbase) {       // called by the elected lane of every warp
        uint64_t* bar = &sm.full[s];
        TileIn<T, kTile>& b = sm.in[s];
        if constexpr (kTable) {
            int64_t rows = nv.table_len - (int64_t)cbase;
            rows = rows < 0 ? 0 : (rows > kNR ? kNR : rows);
            if (cbase < 0) rows = 0;
            sm.nin[s].base = cbase; sm.nin[s].rows = (int32_t)rows;
            if constexpr (TMAP) {           // one box; rows past the end of the table arrive zero-filled and are never read
                mbar_expect_tx(bar, kInBytes + kTile * 4 + (uint32_t)kNR * kTile * 8);
                tensor_load_2d(sm.nin[s].z, &maps.table, (int32_t)i0, cbase < 0 ? 0 : cbase, bar);
            } else {
                mbar_expect_tx(bar, kInBytes + kTile * 4 + (uint32_t)rows * kTile * 8);
                const double* src = nv.table + (int64_t)cbase * nv.table_stride + nv.table_col0 + i0;
                for (int k = 0; k < (int)rows; ++k) bulk_load(sm.nin[s].z[k], src + (int64_t)k * nv.table_stride, kTile * 8, bar);
            }
            bulk_load(sm.nin[s].cursor, st.cursor + i0, kTile * 4, bar);
        } else {
            if (warp == 0) mbar_expect_tx(bar, kInBytes);
        }
        if constexpr (TMAP) {
            tensor_load_2d(b.x, &maps.state, (int32_t)i0, 0, bar);               // x, y, fx, fy, h
        } else {
            if (warp == 0 % kWarps) bulk_load(b.x, st.x + i0, kRow, bar);
            if (warp == 1 % kWarps) bulk_load(b.y, st.y + i0, kRow, bar);
            if (warp == 2 % kWarps) bulk_load(b.fx, st.fx + i0, kRow, bar);
            if (warp == 3 % kWarps) bulk_load(b.fy, st.fy + i0, kRow, bar);
            if (warp == 4 % kWarps) bulk_load(b.h, st.h + i0, kRow, bar);
        }
        if (warp == 5 % kWarps) bulk_load(b.act, act_base + (int64_t)i0 * act_el, act_bytes, bar);
        if (warp == 6 % kWarps) bulk_load(b.counter, ctr_row + i0, kTile * 4, bar);
    };
    // this launch changes a tile's cursors only when it processes the tile, so the elected thread may read the first
    // cursor of a tile it will load later with a plain load, one issue ahead (its latency hides behind a tile)
    auto tile_cursor = [&](uint32_t i0) -> int32_t {
        if constexpr (kTable) { if (i0 < n_full) return st.cursor[i0]; }
        return 0;
    };

    int32_t cb_next = 0;
    const uint32_t first_i0 = (uint32_t)first * kTile;
    if (elect) {
        for (int s = 0; s < kSI; ++s) {
            const uint32_t i0 = first_i0 + s * env_stride;
            if (i0 < n_full) issue_loads(s, i0, tile_cursor(i0));
        }
        cb_next = tile_cursor(first_i0 + kSI * env_stride);
    }

    constexpr bool kPrefetch = MR_RNG_PREFETCH && MODE == MR_NOISE_PHILOX && !MISM;
    auto predraw = [&](uint32_t i0) {                       // this thread's normals for tile i0, parked in shared memory
        if constexpr (kPrefetch) {
            PhiloxNoise nzp;
            nzp.seek(nv.env_base + (uint64_t)(i0 + tid), off);
            float z8[8];
            nzp.draw8(p, z8);
            sm.zpre[tid] = make_float4(z8[0], z8[1], z8[2], z8[3]);
            sm.zpre[kTile + tid] = make_float4(z8[4], z8[5], z8[6], z8[7]);
        }
    };
    if (first_i0 < n_full) predraw(first_i0);

    int s = 0, so = 0;                                      // input / output stage of this tile
    uint32_t parity = 0;                                    // phase of full[s] this tile waits for
    for (uint32_t i0 = first_i0; i0 < n_full; i0 += env_stride) {
        const uint32_t nxt = i0 + kSI * env_stride;         // the tile whose loads re-fill in[s]

        mbar_wait(&sm.full[s], parity);
        Env e;
        const TileIn<T, kTile>& bi = sm.in[s];
        e.x = (double)bi.x[tid]; e.y = (double)bi.y[tid]; e.fx = (double)bi.fx[tid]; e.fy = (double)bi.fy[tid];
        const T h_raw = bi.h[tid];
        e.counter = bi.counter[tid]; e.status = 0; e.spx = e.spy = 0.0;
        double f_t, al;
        if (sizeof(T) == 8 && !act32) { const double2 a2 = reinterpret_cast<const double2*>(bi.act)[tid]; f_t = a2.x; al = a2.y; }
        else { const float2 a2 = reinterpret_cast<const float2*>(bi.act)[tid]; f_t = a2.x; al = a2.y; }

        if constexpr (!kOneBar) {
            if (elect) bulk_wait_read<kStagesOut - 1>();    // out[so] (used kStagesOut tiles ago) has been read out
            __syncthreads();                                // [A] in[s] fully consumed, out[so] free
            if constexpr (!kTable) {
                if (elect && nxt < n_full) issue_loads(s, nxt, 0);
            }
        }

        const double t = time_at(tv, e.counter, p.dt);
        const double tb = t + p.dt, tb2 = tb + p.dt;
        e.h = decode_h<T>(h_raw, tb - t);
        int32_t cur = 0;
        e.counter += 1;                                     // MR_env.py:80
        if constexpr (kTable) {
            TileTableNoise nz;
            nz.stage = &sm.nin[s].z[0][tid]; nz.stage_stride = kTile;
            nz.base = sm.nin[s].base; nz.rows = sm.nin[s].rows;
            nz.col = nv.table + nv.table_col0 + i0 + tid; nz.stride = nv.table_stride;
            nz.cursor = sm.nin[s].cursor[tid]; nz.len = (int32_t)nv.table_len; nz.overflow = 0;
            sim_step<MISM>(e, t, tb, tb2, f_t, al, p, nz);
            cur = nz.cursor;
            if (nz.overflow) e.status |= kNoiseOverflow;
        } else if constexpr (kPrefetch) {
            const float4 za = sm.zpre[tid], zb = sm.zpre[kTile + tid];
            const float z8[8] = {za.x, za.y, za.z, za.w, zb.x, zb.y, zb.z, zb.w};
            if (i0 + env_stride < n_full) predraw(i0 + env_stride);   // independent of everything below
            PhiloxNoise nz;                                     // only the rare multi-attempt path draws from it
            nz.seek(nv.env_base + (uint64_t)(i0 + tid), off);
            nz.blk += 2;
            sim_step_drawn(e, t, tb, tb2, f_t, al, p, nz, z8);
        } else {
            auto nz = make_noise<MODE>(nv, n_total, i0 + tid, 0, off);
            sim_step<MISM>(e, t, tb, tb2, f_t, al, p, nz);
        }
        const Observation o = observe(e, p);
        double d_out = o.d, il_next = tb2 - tb;
        if (auto_reset && o.done) {                         // reported obs = first obs of the new episode
            int ov = 0;
            auto_reset_env<MODE, MISM>(e, nv, n_total, i0 + tid, cur, off, p, ov);
            if (ov) e.status |= kNoiseOverflow;
            d_out = sqrt(e.x * e.x + e.y * e.y);
            il_next = p.dt;
        }

        TileOut<T, kTile>& bo = sm.out[so];
        bo.x[tid] = (T)e.x; bo.y[tid] = (T)e.y; bo.fx[tid] = (T)e.fx; bo.fy[tid] = (T)e.fy;
        bo.h[tid] = encode_h<T>(e.h, il_next);
        bo.counter[tid] = e.counter;
        bo.done[tid] = o.done ? 1 : 0;
        if (out32) {
            // the output-only rows of the stage (d, rew, spx: kTile doubles each) are re-used as 2 * kTile floats:
            // rew <- x | y,  d <- d | rew,  spx <- spx | spy
            float* fxy = reinterpret_cast<float*>(bo.rew); fxy[tid] = (float)e.x; fxy[kTile + tid] = (float)e.y;
            float* fdr = reinterpret_cast<float*>(bo.d); fdr[tid] = (float)d_out; fdr[kTile + tid] = (float)o.rew;
            if (w_sp) { float* fsp = reinterpret_cast<float*>(bo.spx); fsp[tid] = (float)e.spx; fsp[kTile + tid] = (float)e.spy; }
        } else {
            bo.d[tid] = (T)d_out; bo.rew[tid] = (T)o.rew;
            if (w_sp) { bo.spx[tid] = (T)e.spx; bo.spy[tid] = (T)e.spy; }
        }
        if constexpr (kTable) sm.nout[so].cursor[tid] = cur;
        if (e.status) st.status[i0 + tid] |= (uint8_t)e.status;   // rare: sticky flags, plain store
        fence_async_smem();
        __syncthreads();                                    // [B] tile results complete in out[so]
        if (elect) {
            if constexpr (kOneBar) {                        // in[s] was copied to registers before [B] by every thread
                if (nxt < n_full) issue_loads(s, nxt, 0);
            }
            if constexpr (kTable) {                         // the stage's noise rows are free only now
                if (nxt < n_full) issue_loads(s, nxt, cb_next);
                cb_next = tile_cursor(nxt + env_stride);
                bulk_store(st.cursor + i0, sm.nout[so].cursor, kTile * 4);
            }
            if constexpr (TMAP) {
                tensor_store_2d(&maps.state, (int32_t)i0, 0, bo.x);                              // x, y, fx, fy, h
                bulk_store(ctr_row + i0, bo.counter, kTile * 4);
                if (out32) {
                    constexpr uint32_t kRow32 = kTile * 4;
                    const float* fdr = reinterpret_cast<const float*>(bo.d);
                    if (w_obs) {
                        tensor_store_2d(&maps.obs, (int32_t)i0, 0, bo.rew);                      // float x | y
                        if (w_goal) tensor_store_2d(&maps.obs, (int32_t)i0, 2, sm.zero);
                        bulk_store(reinterpret_cast<float*>(out.obs) + 4 * out.stride + i0, fdr, kRow32);
                    }
                    if (w_rew) bulk_store(reinterpret_cast<float*>(out.rew) + i0, fdr + kTile, kRow32);
                    if (w_sp) tensor_store_2d(&maps.sp, (int32_t)i0, 0, bo.spx);                 // float spx | spy
                } else {
                    if (w_obs) {
                        tensor_store_2d(&maps.obs, (int32_t)i0, 0, bo.x);                        // obs rows x, y
                        if (w_goal) tensor_store_2d(&maps.obs, (int32_t)i0, 2, sm.zero);         // goal = (0,0), MR_env.py:57
                        bulk_store(d_row + i0, bo.d, kRow);
                    }
                    if (w_rew) bulk_store(out.rew + i0, bo.rew, kRow);
                    if (w_sp) tensor_store_2d(&maps.sp, (int32_t)i0, 0, bo.spx);
                }
            } else {
            if (warp == 0 % kWarps) bulk_store(st.x + i0, bo.x, kRow);
            if (warp == 1 % kWarps) bulk_store(st.y + i0, bo.y, kRow);
            if (warp == 2 % kWarps) bulk_store(st.fx + i0, bo.fx, kRow);
            if (warp == 3 % kWarps) bulk_store(st.fy + i0, bo.fy, kRow);
            if (warp == 4 % kWarps) bulk_store(st.h + i0, bo.h, kRow);
            if (warp == 5 % kWarps) bulk_store(st.counter + i0, bo.counter, kTile * 4);
            if (out32) {
                constexpr uint32_t kRow32 = kTile * 4;
                float* obs = reinterpret_cast<float*>(out.obs);
                const float* fxy = reinterpret_cast<const float*>(bo.rew);
                const float* fdr = reinterpret_cast<const float*>(bo.d);
                if (obs) {
                    bulk_store(obs + i0, fxy, kRow32);
                    bulk_store(obs + out.stride + i0, fxy + kTile, kRow32);
                    if (out.goal) {
                        bulk_store(obs + 2 * out.stride + i0, sm.zero, kRow32);
                        bulk_store(obs + 3 * out.stride + i0, sm.zero, kRow32);
                    }
                    bulk_store(obs + 4 * out.stride + i0, fdr, kRow32);
                }
                if (out.rew) bulk_store(reinterpret_cast<float*>(out.rew) + i0, fdr + kTile, kRow32);
                if (out.sp) {
                    const float* fsp = reinterpret_cast<const float*>(bo.spx);
                    bulk_store(reinterpret_cast<float*>(out.sp) + i0, fsp, kRow32);
                    bulk_store(reinterpret_cast<float*>(out.sp) + out.stride + i0, fsp + kTile, kRow32);
                }
            } else {
                if (out.obs) {
                    if (warp == 6 % kWarps) bulk_store(out.obs + i0, bo.x, kRow);
                    if (warp == 7 % kWarps) bulk_store(out.obs + out.stride + i0, bo.y, kRow);
                    if (out.goal && warp == 8 % kWarps) bulk_store(out.obs + 2 * out.stride + i0, sm.zero, kRow);   // goal = (0,0), MR_env.py:57
                    if (out.goal && warp == 9 % kWarps) bulk_store(out.obs + 3 * out.stride + i0, sm.zero, kRow);
                    if (warp == 10 % kWarps) bulk_store(out.obs + 4 * out.stride + i0, bo.d, kRow);
                }
                if (out.rew && warp == 11 % kWarps) bulk_store(out.rew + i0, bo.rew, kRow);
                if (out.sp) {
                    if (warp == 13 % kWarps) bulk_store(out.sp + i0, bo.spx, kRow);
                    if (warp == 14 % kWarps) bulk_store(out.sp + out.stride + i0, bo.spy, kRow);
                }
            }
            }
            if (w_done && warp == 12 % kWarps) bulk_store(out.done + i0, bo.done, kTile);
            bulk_commit();                                  // bulk groups are per thread: every issuing lane commits
            if constexpr (kOneBar) bulk_wait_read<1>();     // tile it-1's stores have been read out: frees out[(it + 2) % 3]
        }
        if (++s == kSI) { s = 0; parity ^= 1u; }
        if (++so == kSO) so = 0;
    }
    if (elect) bulk_wait_read<0>();                         // smem must outlive the last bulk stores
}

}  // namespace mr
