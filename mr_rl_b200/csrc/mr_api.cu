// Exported C ABI of the env path (include/mr_rl_b200.h): argument checks and dispatch to the
// per-(storage dtype, noise mode) launchers.  No CPU fallback exists: every call launches CUDA.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <initializer_list>
#include <new>

#include "mr_common.cuh"

namespace mr {

thread_local char g_err[512] = "";

static int step_path_from_env() {
    const char* e = getenv("MR_STEP_PATH");
    if (!e) return 0;
    if (e[0] == 't' && e[1] == 'm' && e[2] == 'a' && e[3] == 'p') return 5;
    return e[0] == 't' ? 1 : e[0] == 'v' ? 2 : e[0] == 's' ? 3 : e[0] == 'w' ? 4 : 0;
}
int g_step_path = step_path_from_env();
thread_local int g_step_cta_cap = 0;
static int actor_path_from_env() {
    const char* e = getenv("MR_ACTOR_PATH");
    return !e ? 0 : e[0] == 's' ? 1 : e[0] == 't' ? 2 : 0;
}
int g_actor_path = actor_path_from_env();

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(MR_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    return MR_OK;
}

static Params to_params(const mr_sim_params& s, const mr_noise* nz) {
    Params p;
    philox_make_keys(nz ? nz->seed : 0, p.keys);
    p.a0 = s.a0; p.sigma = s.noise_var;
    p.dt = s.time_span; p.rtol = s.rtol; p.atol = s.atol;
    p.min_dist = s.min_dist2goal; p.bound_xy = s.bound_xy; p.bound_d = s.bound_d;
    for (int i = 0; i < 2; ++i) { p.init_lo[i] = s.init_low[i]; p.init_hi[i] = s.init_high[i]; p.act_hi[i] = s.action_high[i]; }
    p.mism = s.is_mismatched; p.mism_reset = s.mism_at_reset; p.max_steps = s.max_timesteps;
    p.reward_mode = s.reward_mode; p.auto_reset = s.auto_reset;
    p.act_f32 = s.action_f32;
    finalize_params(p);
    return p;
}

template <class T>
static StateView<T> state_view(const mr_env_state& s) {
    StateView<T> v;
    v.x = (T*)s.x; v.y = (T*)s.y; v.fx = (T*)s.fx; v.fy = (T*)s.fy; v.h = (T*)s.h;
    v.counter = s.counter; v.cursor = s.cursor; v.status = s.status;
    v.a0 = s.a0; v.sigma = s.noise_var; v.mism = s.is_mismatched;
    return v;
}

template <class T>
static OutView<T> out_view(const mr_step_out* o, int64_t n) {
    OutView<T> v;
    v.f32 = false;
    if (!o) { v.obs = nullptr; v.rew = nullptr; v.done = nullptr; v.sp = nullptr; v.stride = n; v.goal = true; return v; }
    v.obs = (T*)o->obs; v.rew = (T*)o->rew; v.done = o->done; v.sp = (T*)o->state_prime;
    v.goal = o->skip_goal_rows == 0;
    v.f32 = sizeof(T) == 8 && o->out_f32 != 0;
    v.stride = o->row_stride ? o->row_stride : n;
    return v;
}

static NoiseView noise_view(const mr_noise* nz, int64_t n) {
    NoiseView v;
    memset(&v, 0, sizeof(v));
    if (nz) {
        v.table = nz->table; v.table_len = nz->table_len; v.seed = nz->seed; v.offset = nz->offset; v.env_base = nz->env_base;
        v.offset_dev = nz->offset_dev;
    }
    v.table_stride = n;        // the table is [table_len][n] for the n envs of this call
    return v;
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

// ---- 2-D TMA tensor maps ------------------------------------------------------------------------------------------
using TmapEncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TmapEncodeFn tmap_encoder() {       // cuTensorMapEncodeTiled through the runtime (no libcuda link)
    static const TmapEncodeFn fn = [] {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) { cudaGetLastError(); ptr = nullptr; }
        return (TmapEncodeFn)ptr;
    }();
    return fn;
}

struct TmapKey { const void* base; uint64_t cols, rows, stride; uint32_t box_cols, box_rows; int dt; };
struct TmapSlot { TmapKey key; CUtensorMap map; bool used; };
static bool tmap_2d(CUtensorMap& out, int dt /*0 f64, 1 f32*/, const void* base, uint64_t cols, uint64_t rows, uint64_t stride_bytes,
                    uint32_t box_cols, uint32_t box_rows) {
    if (!base || !aligned16(base) || (stride_bytes & 15u) || cols == 0 || rows == 0 || box_cols > 256 || box_rows > 256) return false;
    const TmapEncodeFn enc = tmap_encoder();
    if (!enc) return false;
    // the same few tensors are stepped over and over: a tiny per-thread cache keeps the encoder off the launch path
    thread_local TmapSlot cache[16] = {};
    thread_local int next = 0;
    const TmapKey k{base, cols, rows, stride_bytes, box_cols, box_rows, dt};
    for (const TmapSlot& c : cache)
        if (c.used && memcmp(&c.key, &k, sizeof(k)) == 0) { out = c.map; return true; }
    cudaPointerAttributes pa;              // tensor maps over device memory only (host-mapped rows keep the 1-D copies)
    if (cudaPointerGetAttributes(&pa, base) != cudaSuccess || pa.type != cudaMemoryTypeDevice) { cudaGetLastError(); return false; }
    const cuuint64_t gdim[2] = {cols, rows};
    const cuuint64_t gstr[1] = {stride_bytes};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t es[2] = {1, 1};
    CUtensorMap m;
    const CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_NONE;   // 128 B / 256 B promotion measured: no difference
    const CUresult r = enc(&m, dt == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), gdim,
                           gstr, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, promo,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
    TmapSlot& slot = cache[next];
    next = (next + 1) % 16;
    memset(&slot.key, 0, sizeof(slot.key));
    slot.key = k; slot.map = m; slot.used = true;
    out = m;
    return true;
}

template <class T>
bool build_step_maps(StepMaps& m, const StateView<T>& sv, const OutView<T>& ov, const NoiseView& nv, int64_t n, int tile,
                     int table_rows) {
    memset(&m, 0, sizeof(m));
    const int dt = sizeof(T) == 8 ? 0 : 1;
    const ptrdiff_t stride = (const char*)sv.y - (const char*)sv.x;       // x, y, fx, fy, h equally strided?
    if (stride <= 0 || (const char*)sv.fx - (const char*)sv.y != stride || (const char*)sv.fy - (const char*)sv.fx != stride ||
        (const char*)sv.h - (const char*)sv.fy != stride || stride < (ptrdiff_t)(n * sizeof(T)))
        return false;
    if (!tmap_2d(m.state, dt, sv.x, (uint64_t)n, 5, (uint64_t)stride, (uint32_t)tile, 5)) return false;
    const int dt_out = (sizeof(T) == 8 && !ov.f32) ? 0 : 1;
    const uint64_t el_out = dt_out == 0 ? 8 : 4;
    if (ov.obs && !tmap_2d(m.obs, dt_out, ov.obs, (uint64_t)n, 5, (uint64_t)ov.stride * el_out, (uint32_t)tile, 2)) return false;
    if (ov.sp && !tmap_2d(m.sp, dt_out, ov.sp, (uint64_t)n, 2, (uint64_t)ov.stride * el_out, (uint32_t)tile, 2)) return false;
    if (table_rows > 0) {
        if (nv.table_col0 != 0) return false;
        if (!tmap_2d(m.table, 0, nv.table, (uint64_t)nv.table_stride, (uint64_t)nv.table_len, (uint64_t)nv.table_stride * 8,
                     (uint32_t)tile, (uint32_t)table_rows))
            return false;
    }
    return true;
}
template bool build_step_maps<double>(StepMaps&, const StateView<double>&, const OutView<double>&, const NoiseView&, int64_t, int, int);
template bool build_step_maps<float>(StepMaps&, const StateView<float>&, const OutView<float>&, const NoiseView&, int64_t, int, int);

// every row the vectorised step kernel touches must start on a 16-byte boundary
template <class T>
static bool rows_aligned(const mr_env_state& s, const mr_step_out* o, const void* actions, int64_t n) {
    bool ok = aligned16(s.x) && aligned16(s.y) && aligned16(s.fx) && aligned16(s.fy) && aligned16(s.h) &&
              aligned16(s.counter) && aligned16(actions);
    if (o) {
        const int64_t stride = o->row_stride ? o->row_stride : n;
        const int64_t el_out = o->out_f32 ? 4 : (int64_t)sizeof(T);
        const bool stride_ok = (stride * el_out) % 16 == 0;
        if (o->obs) ok = ok && aligned16(o->obs) && stride_ok;
        if (o->state_prime) ok = ok && aligned16(o->state_prime) && stride_ok;
        if (o->rew) ok = ok && aligned16(o->rew);
        if (o->done) ok = ok && aligned16(o->done);
    }
    return ok;
}

static int check_common(const char* fn, const mr_env_state* st, int64_t n, int dtype, const mr_sim_params* p, const mr_noise* nz) {
    if (!st || !p) return fail(MR_ERR_ARG, "%s: null state/params", fn);
    if (n < 0 || n > ((int64_t)1 << 31) - 1) return fail(MR_ERR_ARG, "%s: bad n=%lld", fn, (long long)n);
    if (dtype != MR_F64 && dtype != MR_F32) return fail(MR_ERR_ARG, "%s: bad dtype %d", fn, dtype);
    if (n > 0 && (!st->x || !st->y || !st->fx || !st->fy || !st->h || !st->counter || !st->status))
        return fail(MR_ERR_ARG, "%s: null state row", fn);
    const int mode = nz ? nz->mode : MR_NOISE_NONE;
    if (mode != MR_NOISE_NONE && mode != MR_NOISE_TABLE && mode != MR_NOISE_PHILOX)
        return fail(MR_ERR_ARG, "%s: unknown noise mode %d", fn, mode);
    if (mode == MR_NOISE_TABLE) {
        if (!nz->table || nz->table_len <= 0) return fail(MR_ERR_ARG, "%s: table noise without a table", fn);
        if (!st->cursor) return fail(MR_ERR_ARG, "%s: table noise needs state.cursor", fn);
    }
    if (mode == MR_NOISE_NONE && p->noise_var != 0.0 && !st->noise_var)
        return fail(MR_ERR_ARG, "%s: noise_var=%g needs a noise source (table or philox)", fn, p->noise_var);
    const int rows = (st->a0 != nullptr) + (st->noise_var != nullptr) + (st->is_mismatched != nullptr);
    if (rows != 0 && rows != 3) return fail(MR_ERR_ARG, "%s: give all three per-env parameter rows (a0, noise_var, is_mismatched) or none", fn);
    if (!(p->time_span > 0.0)) return fail(MR_ERR_ARG, "%s: time_span must be positive", fn);
    return MR_OK;
}

template <class T>
static int do_step(const mr_env_state& st, int64_t n, const Params& p, const mr_noise* nz, const TimeView& tv,
                   const void* actions, const mr_step_out* out, cudaStream_t s) {
    const StateView<T> sv = state_view<T>(st);
    const OutView<T> ov = out_view<T>(out, n);
    const NoiseView nv = noise_view(nz, n);
    bool vec_ok = rows_aligned<T>(st, out, actions, n);
    if (nz && nz->mode == MR_NOISE_TABLE)      // bulk copies of table rows: every row of the tile must be 16-byte aligned
        vec_ok = vec_ok && aligned16(nz->table) && n % 2 == 0 && aligned16(st.cursor);
    switch (nz ? nz->mode : MR_NOISE_NONE) {
        case MR_NOISE_TABLE: return launch_step<T, MR_NOISE_TABLE>(sv, (const T*)actions, ov, nv, tv, p, n, vec_ok, s);
        case MR_NOISE_PHILOX: return launch_step<T, MR_NOISE_PHILOX>(sv, (const T*)actions, ov, nv, tv, p, n, vec_ok, s);
        default: return launch_step<T, MR_NOISE_NONE>(sv, (const T*)actions, ov, nv, tv, p, n, vec_ok, s);
    }
}

template <class T>
static int do_reset(const mr_env_state& st, int64_t n, const Params& p, const mr_noise* nz, const void* init_xy,
                    const uint8_t* mask, int reset_cursor, const mr_reset_params* rp, const mr_step_out* out, cudaStream_t s) {
    const StateView<T> sv = state_view<T>(st);
    const OutView<T> ov = out_view<T>(out, n);
    const NoiseView nv = noise_view(nz, n);
    ResetRows rr{nullptr, nullptr, nullptr};
    if (rp) { rr.a0 = rp->a0; rr.sigma = rp->noise_var; rr.mism = rp->is_mismatched; }
    switch (nz ? nz->mode : MR_NOISE_NONE) {
        case MR_NOISE_TABLE: return launch_reset<T, MR_NOISE_TABLE>(sv, (const T*)init_xy, mask, reset_cursor, rr, ov, nv, p, n, s);
        case MR_NOISE_PHILOX: return launch_reset<T, MR_NOISE_PHILOX>(sv, (const T*)init_xy, mask, reset_cursor, rr, ov, nv, p, n, s);
        default: return launch_reset<T, MR_NOISE_NONE>(sv, (const T*)init_xy, mask, reset_cursor, rr, ov, nv, p, n, s);
    }
}

__global__ void counter_set_kernel(uint64_t* c, uint64_t v) { *c = v; }

// the standard normals of one Philox stream, in the order PhiloxNoise::next() / draw8() hand them out
struct KeysOnly { PhiloxKeys keys; };
__global__ void philox_normals_kernel(KeysOnly k, uint64_t env_base, uint64_t step, uint32_t purpose, int count, int64_t n,
                                      float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    PhiloxNoise nz;
    nz.seek(env_base + (uint64_t)i, step, purpose);
    for (int j = 0; j < count; ++j) out[(int64_t)j * n + i] = (float)nz.next(k);
}

template <class T>
static RolloutView<T> rollout_view(const mr_rollout_io& io) {
    RolloutView<T> rv;
    rv.actions = (const T*)io.actions; rv.actor = io.actor; rv.traj_xy = (T*)io.traj_xy;
    rv.traj_sp = (T*)io.traj_state_prime; rv.traj_done = io.traj_done; rv.stats = io.stats;
    rv.traj_actions = (T*)io.traj_actions; rv.traj_rew = (T*)io.traj_rew; rv.traj_reset_xy = (T*)io.traj_reset_xy;
    rv.traj_episode = io.traj_episode; rv.traj_step = io.traj_step; rv.episode_counter = io.episode_counter;
    rv.reset_init = (const T*)io.reset_init; rv.reset_init_len = io.reset_init_len;
    rv.k_steps = io.k_steps; rv.action_source = io.action_source;
    return rv;
}

template <class T>
static int do_rollout(const mr_env_state& st, int64_t n, const Params& p, const mr_noise* nz, const TimeView& tv,
                      const mr_rollout_io& io, const GpHeadingView* gh, const CollectView* cv, const mr_step_out* out,
                      cudaStream_t s) {
    const RolloutView<T> rv = rollout_view<T>(io);
    const StateView<T> sv = state_view<T>(st);
    const OutView<T> ov = out_view<T>(out, n);
    const NoiseView nv = noise_view(nz, n);
    switch (nz ? nz->mode : MR_NOISE_NONE) {
        case MR_NOISE_TABLE: return launch_rollout<T, MR_NOISE_TABLE>(sv, rv, ov, nv, tv, p, n, gh, cv, nullptr, s);
        case MR_NOISE_PHILOX: return launch_rollout<T, MR_NOISE_PHILOX>(sv, rv, ov, nv, tv, p, n, gh, cv, nullptr, s);
        default: return launch_rollout<T, MR_NOISE_NONE>(sv, rv, ov, nv, tv, p, n, gh, cv, nullptr, s);
    }
}

// the checks of mr_env_rollout that do not depend on the action source
static int check_rollout(const char* fn, const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                         const mr_noise* nz, const mr_rollout_io* io, const mr_step_out* out) {
    int rc = check_common(fn, st, n, dtype, p, nz);
    if (rc) return rc;
    if (!io || io->k_steps < 0) return fail(MR_ERR_ARG, "%s: bad io", fn);
    if (p->auto_reset && nz == nullptr) return fail(MR_ERR_ARG, "%s: auto_reset needs mr_noise (seed) for the init sampler", fn);
    if (out && out->out_f32) return fail(MR_ERR_UNSUPPORTED, "%s: float32 output rows are a step option", fn);
    if (io->reset_init && io->reset_init_len <= 0) return fail(MR_ERR_ARG, "%s: reset_init needs reset_init_len > 0", fn);
    return MR_OK;
}

}  // namespace mr

extern "C" {

int mr_abi_version(void) { return MR_ABI_VERSION; }
const char* mr_last_error(void) { return mr::g_err; }

int mr_set_step_path(int32_t path) {
    if (path < 0 || path > 5) return mr::fail(MR_ERR_ARG, "mr_set_step_path: path must be 0..5");
    const int old = mr::g_step_path;
    mr::g_step_path = path;
    return old;
}

int mr_set_actor_path(int32_t path) {
    if (path < 0 || path > 2) return mr::fail(MR_ERR_ARG, "mr_set_actor_path: path must be 0..2");
    const int old = mr::g_actor_path;
    mr::g_actor_path = path;
    return old;
}

void mr_default_params(mr_sim_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->a0 = 1.0; p->noise_var = 1.0;                 /* MR_Env.reset defaults, MR_env.py:167-168 */
    p->time_span = 0.030; p->rtol = 0.030 / 100; p->atol = 1e-4;   /* MR_simulator.py:12-13,91 */
    p->max_timesteps = 50; p->min_dist2goal = 30;    /* MR_env.py:62-63 */
    p->bound_xy = 5000; p->bound_d = 80000;          /* MR_env.py:37-39 */
    p->init_low[0] = p->init_low[1] = 100; p->init_high[0] = p->init_high[1] = 120;   /* :40-42 */
    p->action_high[0] = 20; p->action_high[1] = 2 * 3.141592653589793;                /* :34-36 */
}

void mr_fill_time_table_host(double* t, int32_t len, double time_span) {
    if (!t || len <= 0) return;
    t[0] = 0.0;
    for (int32_t k = 1; k < len; ++k) t[k] = t[k - 1] + time_span;
}

int mr_env_reset_ex(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p, const mr_noise* nz,
                    const void* init_xy, const uint8_t* mask, int32_t reset_cursor, const mr_reset_params* rp,
                    const mr_step_out* out, void* stream) {
    mr::NvtxRange nvtx_range("mr_env_reset_ex");
    int rc = mr::check_common("mr_env_reset", st, n, dtype, p, nz);
    if (rc) return rc;
    if (rp && (rp->a0 || rp->noise_var || rp->is_mismatched) && !st->a0)
        return mr::fail(MR_ERR_ARG, "mr_env_reset: per-env reset arguments need the per-env parameter rows in the state");
    if (out && out->out_f32) return mr::fail(MR_ERR_UNSUPPORTED, "mr_env_reset: float32 output rows are a step option");
    if (n == 0) return MR_OK;
    const mr::Params pp = mr::to_params(*p, nz);
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == MR_F64 ? mr::do_reset<double>(*st, n, pp, nz, init_xy, mask, reset_cursor, rp, out, s)
                           : mr::do_reset<float>(*st, n, pp, nz, init_xy, mask, reset_cursor, rp, out, s);
}

int mr_env_reset(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p, const mr_noise* nz,
                 const void* init_xy, const uint8_t* mask, int32_t reset_cursor, const mr_step_out* out, void* stream) {
    return mr_env_reset_ex(st, n, dtype, p, nz, init_xy, mask, reset_cursor, nullptr, out, stream);
}

int mr_counter_set(uint64_t* counter_dev, uint64_t value, void* stream) {
    if (!counter_dev) return mr::fail(MR_ERR_ARG, "mr_counter_set: null counter");
    mr::counter_set_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter_dev, value);
    return mr::check_launch("mr_counter_set");
}

int mr_env_step(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p, const mr_noise* nz,
                const mr_time_table* tt, const void* actions, const mr_step_out* out, void* stream) {
    mr::NvtxRange nvtx_range("mr_env_step");
    int rc = mr::check_common("mr_env_step", st, n, dtype, p, nz);
    if (rc) return rc;
    if (n == 0) return MR_OK;
    if (!actions) return mr::fail(MR_ERR_ARG, "mr_env_step: null actions");
    if (!tt || !tt->t || tt->len < 2) return mr::fail(MR_ERR_ARG, "mr_env_step: time table missing");
    const mr::Params pp = mr::to_params(*p, nz);
    mr::TimeView tv{tt->t, tt->len};
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == MR_F64 ? mr::do_step<double>(*st, n, pp, nz, tv, actions, out, s)
                           : mr::do_step<float>(*st, n, pp, nz, tv, actions, out, s);
}

// ---- MR_Env.step with HOST buffers: the pipelined H2D -> step -> D2H path in one call ------------------------------
struct mr_host_pipeline {
    int device;
    int max_chunks;
    cudaStream_t s_in, s_k, s_out;
    cudaEvent_t ev_start, ev_done;
    cudaEvent_t* ev_in;      // [max_chunks]
    cudaEvent_t* ev_k;       // [max_chunks]
};

int mr_host_pipeline_create(int32_t max_chunks, mr_host_pipeline** out) {
    if (!out || max_chunks < 1 || max_chunks > 64) return mr::fail(MR_ERR_ARG, "mr_host_pipeline_create: need 1 <= max_chunks <= 64");
    *out = nullptr;
    mr_host_pipeline* pl = new (std::nothrow) mr_host_pipeline();    // value-initialised: every handle starts null
    if (!pl) return mr::fail(MR_ERR_CUDA, "mr_host_pipeline_create: out of host memory");
    pl->max_chunks = max_chunks;
    cudaGetDevice(&pl->device);
    pl->ev_in = new (std::nothrow) cudaEvent_t[max_chunks]();
    pl->ev_k = new (std::nothrow) cudaEvent_t[max_chunks]();
    if (!pl->ev_in || !pl->ev_k) {
        mr_host_pipeline_destroy(pl);
        return mr::fail(MR_ERR_CUDA, "mr_host_pipeline_create: out of host memory");
    }
    cudaError_t e = cudaStreamCreateWithFlags(&pl->s_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&pl->s_k, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&pl->s_out, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&pl->ev_start, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&pl->ev_done, cudaEventDisableTiming);
    for (int i = 0; i < max_chunks && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&pl->ev_in[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&pl->ev_k[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        mr_host_pipeline_destroy(pl);                                // frees whatever was created so far
        return mr::fail(MR_ERR_CUDA, "mr_host_pipeline_create: %s", cudaGetErrorString(e));
    }
    *out = pl;
    return MR_OK;
}

void mr_host_pipeline_destroy(mr_host_pipeline* pl) {
    if (!pl) return;
    if (pl->s_in) cudaStreamDestroy(pl->s_in);
    if (pl->s_k) cudaStreamDestroy(pl->s_k);
    if (pl->s_out) cudaStreamDestroy(pl->s_out);
    if (pl->ev_start) cudaEventDestroy(pl->ev_start);
    if (pl->ev_done) cudaEventDestroy(pl->ev_done);
    for (int i = 0; i < pl->max_chunks; ++i) {
        if (pl->ev_in && pl->ev_in[i]) cudaEventDestroy(pl->ev_in[i]);
        if (pl->ev_k && pl->ev_k[i]) cudaEventDestroy(pl->ev_k[i]);
    }
    delete[] pl->ev_in; delete[] pl->ev_k;
    delete pl;
}

int mr_env_step_host(mr_host_pipeline* pl, const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                     const mr_noise* nz, const mr_time_table* tt, const mr_host_step_io* io, const mr_step_out* out_dev,
                     int32_t n_chunks, void* stream) {
    mr::NvtxRange nvtx_range("mr_env_step_host");
    int rc = mr::check_common("mr_env_step_host", st, n, dtype, p, nz);
    if (rc) return rc;
    if (!io) return mr::fail(MR_ERR_ARG, "mr_env_step_host: null io");
    if (!io->actions_host || !io->obs_host || !io->done_host)
        return mr::fail(MR_ERR_ARG, "mr_env_step_host: null host buffer");
    if (io->io_f32 && (n_chunks != 0 || dtype != MR_F64))
        return mr::fail(MR_ERR_ARG, "mr_env_step_host: io_f32 is the direct mode (n_chunks = 0) with MR_F64 storage");
    if (n == 0) return MR_OK;
    const int64_t el = dtype == MR_F64 ? 8 : 4;
    const int64_t hstride = io->host_row_stride ? io->host_row_stride : n;
    if (n_chunks == 0) {
        // direct mode: the step kernel itself reads the actions from and writes obs / rew / done to the page-locked
        // host buffers (device-addressable under unified addressing) — its TMA bulk copies go over PCIe in both
        // directions at once, there is no staging pass, no per-copy latency and the goal rows are never sent
        mr_step_out oh;
        oh.obs = io->obs_host; oh.rew = io->rew_host; oh.done = io->done_host;
        oh.state_prime = out_dev ? out_dev->state_prime : nullptr;
        oh.row_stride = hstride;
        if (oh.state_prime && (out_dev->row_stride ? out_dev->row_stride : n) != hstride)
            return mr::fail(MR_ERR_ARG, "mr_env_step_host: direct mode shares one row stride between obs_host and state_prime");
        oh.skip_goal_rows = io->copy_goal_rows ? 0 : 1;
        oh.out_f32 = io->io_f32 ? 1 : 0;
        mr_sim_params ph = *p;
        if (io->io_f32) { ph.action_f32 = 1; oh.state_prime = nullptr; }   // float32 host rows; state_prime stays on the device side
        mr::g_step_cta_cap = 1;                         // PCIe-bound: one CTA per SM (see launch_persistent)
        rc = mr_env_step(st, n, dtype, &ph, nz, tt, io->actions_host, &oh, stream);
        mr::g_step_cta_cap = 0;
        if (rc) return rc;
        const cudaError_t e0 = cudaStreamSynchronize((cudaStream_t)stream);
        if (e0 != cudaSuccess) return mr::fail(MR_ERR_CUDA, "mr_env_step_host: %s", cudaGetErrorString(e0));
        return MR_OK;
    }
    if (!pl || !out_dev) return mr::fail(MR_ERR_ARG, "mr_env_step_host: staged mode needs a pipeline and device output rows");
    // actions_dev == NULL: the chunk kernels read the page-locked actions themselves (no H2D copies), only the results
    // go through the copy engine
    const bool zc_in = io->actions_dev == nullptr;
    if (!out_dev->obs || !out_dev->rew || !out_dev->done) return mr::fail(MR_ERR_ARG, "mr_env_step_host: device obs/rew/done rows required");
    const int64_t dstride = out_dev->row_stride ? out_dev->row_stride : n;
    // chunk edges are multiples of 256 envs (tile- and 16-byte aligned sub-ranges); table noise indexes the table by
    // the launch-local env index, so it stays in one piece
    int chunks = n_chunks < 1 ? 1 : (n_chunks > pl->max_chunks ? pl->max_chunks : n_chunks);
    if (nz && nz->mode == MR_NOISE_TABLE) chunks = 1;
    int64_t per = (n / chunks) / 256 * 256;
    if (per == 0) { chunks = 1; per = n; }
    cudaStream_t cur = (cudaStream_t)stream;
    // every asynchronous call is checked; after a failure nothing more is queued, but the caller's stream is still
    // joined to the internal streams below, so no work of this call is left running behind the caller's back
    cudaError_t ce = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (ce == cudaSuccess && r != cudaSuccess) ce = r; return ce == cudaSuccess; };
    ok(cudaEventRecord(pl->ev_start, cur));
    ok(cudaStreamWaitEvent(pl->s_in, pl->ev_start, 0));
    ok(cudaStreamWaitEvent(pl->s_k, pl->ev_start, 0));
    ok(cudaStreamWaitEvent(pl->s_out, pl->ev_start, 0));
    for (int c = 0; c < chunks && ce == cudaSuccess && rc == MR_OK; ++c) {
        const int64_t lo = c * per, hi = c == chunks - 1 ? n : lo + per, m = hi - lo;
        if (!zc_in) {
            if (!ok(cudaMemcpyAsync((char*)io->actions_dev + 2 * lo * el, (const char*)io->actions_host + 2 * lo * el,
                                    (size_t)(2 * m * el), cudaMemcpyHostToDevice, pl->s_in))) break;
            if (!ok(cudaEventRecord(pl->ev_in[c], pl->s_in)) || !ok(cudaStreamWaitEvent(pl->s_k, pl->ev_in[c], 0))) break;
        }
        mr_env_state sc = *st;
        sc.x = (char*)st->x + lo * el; sc.y = (char*)st->y + lo * el; sc.fx = (char*)st->fx + lo * el;
        sc.fy = (char*)st->fy + lo * el; sc.h = (char*)st->h + lo * el;
        sc.counter = st->counter + lo; sc.status = st->status + lo;
        if (st->cursor) sc.cursor = st->cursor + lo;
        mr_step_out oc = *out_dev;
        oc.obs = (char*)out_dev->obs + lo * el; oc.rew = (char*)out_dev->rew + lo * el; oc.done = out_dev->done + lo;
        if (out_dev->state_prime) oc.state_prime = (char*)out_dev->state_prime + lo * el;
        oc.row_stride = dstride;
        mr_noise nc;
        const mr_noise* nzp = nz;
        if (nz) { nc = *nz; nc.env_base = nz->env_base + (uint64_t)lo; nzp = &nc; }
        rc = mr_env_step(&sc, m, dtype, p, nzp, tt, (const char*)(zc_in ? io->actions_host : io->actions_dev) + 2 * lo * el, &oc,
                         pl->s_k);
        if (rc) break;                                              // joined and reported below
        if (!ok(cudaEventRecord(pl->ev_k[c], pl->s_k)) || !ok(cudaStreamWaitEvent(pl->s_out, pl->ev_k[c], 0))) break;
        // rows x, y (and the goal rows, if wanted) are equally pitched: one 2-D copy; then d
        ok(cudaMemcpy2DAsync((char*)io->obs_host + lo * el, (size_t)(hstride * el), (const char*)out_dev->obs + lo * el,
                             (size_t)(dstride * el), (size_t)(m * el), io->copy_goal_rows ? 4 : 2, cudaMemcpyDeviceToHost, pl->s_out));
        ok(cudaMemcpyAsync((char*)io->obs_host + (4 * hstride + lo) * el, (const char*)out_dev->obs + (4 * dstride + lo) * el,
                           (size_t)(m * el), cudaMemcpyDeviceToHost, pl->s_out));
        if (io->rew_host)                                               // NULL: the constant reward of MR_env.py:89 is not sent
            ok(cudaMemcpyAsync((char*)io->rew_host + lo * el, (const char*)out_dev->rew + lo * el, (size_t)(m * el),
                               cudaMemcpyDeviceToHost, pl->s_out));
        ok(cudaMemcpyAsync(io->done_host + lo, out_dev->done + lo, (size_t)m, cudaMemcpyDeviceToHost, pl->s_out));
    }
    // join: later work on the caller's stream sees the new state; the host buffers are valid when s_out has drained
    const cudaError_t j0 = cudaEventRecord(pl->ev_done, pl->s_k);
    const cudaError_t j1 = j0 == cudaSuccess ? cudaStreamWaitEvent(cur, pl->ev_done, 0) : j0;
    const cudaError_t j2 = cudaStreamSynchronize(pl->s_in);
    const cudaError_t j3 = cudaStreamSynchronize(pl->s_out);
    if (rc) return rc;                                              // mr_env_step already set the message
    for (cudaError_t e : {ce, j1, j2, j3})
        if (e != cudaSuccess) return mr::fail(MR_ERR_CUDA, "mr_env_step_host: %s", cudaGetErrorString(e));
    return mr::check_launch("mr_env_step_host");
}

int mr_philox_normals(uint64_t seed, uint64_t env_base, uint64_t step, int32_t stream_id, int32_t count, int64_t n, float* z_out,
                      void* stream) {
    if (!z_out || n < 0 || count < 0 || (stream_id != 0 && stream_id != 1))
        return mr::fail(MR_ERR_ARG, "mr_philox_normals: bad argument");
    if (n == 0 || count == 0) return MR_OK;
    mr::KeysOnly k;
    mr::philox_make_keys(seed, k.keys);
    const uint32_t purpose = stream_id == 0 ? mr::kPurposeNoise : mr::kPurposeResetNoise;
    mr::philox_normals_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(k, env_base, step, purpose, count, n, z_out);
    return mr::check_launch("mr_philox_normals");
}

int mr_host_register(void* host_ptr, int64_t bytes) {
    if (!host_ptr || bytes <= 0) return mr::fail(MR_ERR_ARG, "mr_host_register: null pointer or empty range");
    int dev = 0, same = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&same, cudaDevAttrCanUseHostPointerForRegisteredMem, dev);
    if (!same) return mr::fail(MR_ERR_UNSUPPORTED, "mr_host_register: this platform needs a separate device pointer for registered memory");
    const cudaError_t e = cudaHostRegister(host_ptr, (size_t)bytes, cudaHostRegisterDefault);
    if (e != cudaSuccess) { cudaGetLastError(); return mr::fail(MR_ERR_CUDA, "mr_host_register: %s", cudaGetErrorString(e)); }
    return MR_OK;
}

int mr_host_unregister(void* host_ptr) {
    const cudaError_t e = cudaHostUnregister(host_ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return mr::fail(MR_ERR_CUDA, "mr_host_unregister: %s", cudaGetErrorString(e)); }
    return MR_OK;
}

int mr_env_rollout(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p, const mr_noise* nz,
                   const mr_time_table* tt, const mr_rollout_io* io, const mr_step_out* out, void* stream) {
    mr::NvtxRange nvtx_range("mr_env_rollout");
    int rc = mr::check_common("mr_env_rollout", st, n, dtype, p, nz);
    if (rc) return rc;
    if (!io || io->k_steps < 0) return mr::fail(MR_ERR_ARG, "mr_env_rollout: bad io");
    if (n == 0 || io->k_steps == 0) return MR_OK;
    if (!tt || !tt->t || tt->len < 2) return mr::fail(MR_ERR_ARG, "mr_env_rollout: time table missing");
    if (io->action_source < 0 || io->action_source > MR_ACTIONS_BROADCAST)
        return mr::fail(MR_ERR_ARG, "mr_env_rollout: unknown action source %d", io->action_source);
    if ((io->action_source == MR_ACTIONS_TENSOR || io->action_source == MR_ACTIONS_BROADCAST) && !io->actions)
        return mr::fail(MR_ERR_ARG, "mr_env_rollout: null actions");
    if (io->action_source == MR_ACTIONS_ACTOR && !io->actor) return mr::fail(MR_ERR_ARG, "mr_env_rollout: null actor");
    if (io->action_source == MR_ACTIONS_TENSOR && !mr::aligned16(io->actions))
        return mr::fail(MR_ERR_ARG, "mr_env_rollout: actions must be 16-byte aligned");
    if (p->auto_reset && nz == nullptr)
        return mr::fail(MR_ERR_ARG, "mr_env_rollout: auto_reset needs mr_noise (seed) for the init sampler");
    if (out && out->out_f32) return mr::fail(MR_ERR_UNSUPPORTED, "mr_env_rollout: float32 output rows are a step option");
    if (io->reset_init && io->reset_init_len <= 0) return mr::fail(MR_ERR_ARG, "mr_env_rollout: reset_init needs reset_init_len > 0");
    if (p->action_f32 && dtype == MR_F64 && io->action_source == MR_ACTIONS_TENSOR)
        return mr::fail(MR_ERR_UNSUPPORTED, "mr_env_rollout: float32 actions with fp64 storage are a step option");
    const mr::Params pp = mr::to_params(*p, nz);
    mr::TimeView tv{tt->t, tt->len};
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == MR_F64 ? mr::do_rollout<double>(*st, n, pp, nz, tv, *io, nullptr, nullptr, out, s)
                           : mr::do_rollout<float>(*st, n, pp, nz, tv, *io, nullptr, nullptr, out, s);
}

}  // extern "C"

extern "C" int mr_env_rollout_gp_heading(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                                         const mr_noise* nz, const mr_time_table* tt, const mr_rollout_io* io,
                                         const mr_gp_heading_policy* pol, const mr_step_out* out, void* stream) {
    mr::NvtxRange nvtx_range("mr_env_rollout_gp_heading");
    using mr::fail;
    const char* fn = "mr_env_rollout_gp_heading";
    int rc = mr::check_rollout(fn, st, n, dtype, p, nz, io, out);
    if (rc) return rc;
    if (io->action_source != MR_ACTIONS_GP_HEADING)
        return fail(MR_ERR_ARG, "%s: io->action_source must be MR_ACTIONS_GP_HEADING (%d), got %d", fn, MR_ACTIONS_GP_HEADING,
                    io->action_source);
    if (!pol) return fail(MR_ERR_ARG, "%s: null policy", fn);
    if (!pol->coef_x || !pol->coef_y) return fail(MR_ERR_ARG, "%s: null coefficients", fn);
    if (!pol->ref) return fail(MR_ERR_ARG, "%s: null ref", fn);
    if (pol->n_coef < 1 || pol->n_coef > 4096) return fail(MR_ERR_ARG, "%s: need 1 <= n_coef <= 4096", fn);
    for (double v : {pol->a0, pol->freq, pol->drift_x, pol->drift_y, pol->gain})
        if (!std::isfinite(v)) return fail(MR_ERR_ARG, "%s: a0, freq, drift_x, drift_y and gain must be finite", fn);
    if (st->a0) return fail(MR_ERR_UNSUPPORTED, "%s: the GP heading policy does not take per-env parameter rows", fn);
    if (n == 0 || io->k_steps == 0) return MR_OK;
    if (!tt || !tt->t || tt->len < 2) return fail(MR_ERR_ARG, "%s: time table missing", fn);
    const mr::Params pp = mr::to_params(*p, nz);
    const mr::TimeView tv{tt->t, tt->len};
    mr::GpHeadingView gh;
    gh.coef_x = pol->coef_x; gh.coef_y = pol->coef_y; gh.ref = pol->ref;
    gh.a0f = pol->a0 * pol->freq;                           // as mr_gp_correct_heading_cheb forms it
    gh.dx = pol->drift_x; gh.dy = pol->drift_y;
    gh.freq = pol->freq; gh.gain = pol->gain;
    gh.lo = -3.141592653589793; gh.hi = 3.141592653589793; gh.xatol = 1e-5;
    gh.n_coef = pol->n_coef; gh.maxfun = 500;
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == MR_F64 ? mr::do_rollout<double>(*st, n, pp, nz, tv, *io, &gh, nullptr, out, s)
                           : mr::do_rollout<float>(*st, n, pp, nz, tv, *io, &gh, nullptr, out, s);
}

namespace mr {
// the checks of mr_env_rollout_ddpg_collect, and its CollectView; ring_envs: the envs that write into one ring (n, or a
// population member's N), described by `what` in the error message
static int collect_view(const char* fn, const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                        const mr_noise* nz, const mr_time_table* tt, const mr_rollout_io* io, const mr_ddpg_collect* c,
                        const mr_step_out* out, int64_t ring_envs, const char* what, CollectView& cv) {
    int rc = check_rollout(fn, st, n, dtype, p, nz, io, out);
    if (rc) return rc;
    if (io->action_source != MR_ACTIONS_ACTOR)
        return fail(MR_ERR_ARG, "%s: io->action_source must be MR_ACTIONS_ACTOR (%d), got %d", fn, MR_ACTIONS_ACTOR, io->action_source);
    if (!io->actor) return fail(MR_ERR_ARG, "%s: null actor", fn);
    if (!c) return fail(MR_ERR_ARG, "%s: null collect struct", fn);
    if (!c->ou_state) return fail(MR_ERR_ARG, "%s: null ou_state", fn);
    const mr_replay& rb = c->ring;
    if (!rb.s || !rb.a || !rb.r || !rb.d || !rb.s2) return fail(MR_ERR_ARG, "%s: null replay ring array", fn);
    if (!out || !out->obs) return fail(MR_ERR_ARG, "%s: the observation rows out->obs (the first policy input) are required", fn);
    if (rb.capacity <= 0) return fail(MR_ERR_ARG, "%s: ring capacity must be positive", fn);
    if (c->head < 0 || c->head >= rb.capacity) return fail(MR_ERR_ARG, "%s: need 0 <= head < capacity", fn);
    if (ring_envs > rb.capacity) return fail(MR_ERR_ARG, "%s: %s", fn, what);
    for (double v : {c->ou_theta, c->ou_mu, c->ou_sigma, c->ou_dt})
        if (!std::isfinite(v)) return fail(MR_ERR_ARG, "%s: ou_theta, ou_mu, ou_sigma and ou_dt must be finite", fn);
    if (!tt || !tt->t || tt->len < 2) return fail(MR_ERR_ARG, "%s: time table missing", fn);
    if (st->a0) return fail(MR_ERR_UNSUPPORTED, "%s: the collector does not take per-env parameter rows", fn);
    if (g_actor_path == 1) return fail(MR_ERR_UNSUPPORTED, "%s: the CUDA-core actor path (mr_set_actor_path(1)) has no collector", fn);
    cv.ou = c->ou_state;
    philox_make_keys(c->ou_seed, cv.keys);
    cv.theta = c->ou_theta; cv.mu = c->ou_mu; cv.sd = c->ou_sigma * sqrt(c->ou_dt); cv.dt = c->ou_dt;
    cv.counter = c->ou_counter; cv.env_base = c->ou_env_base;
    cv.s = rb.s; cv.a = rb.a; cv.r = rb.r; cv.d = rb.d; cv.s2 = rb.s2;
    cv.capacity = rb.capacity; cv.head = c->head;
    cv.member_envs = 0;
    return MR_OK;
}
}  // namespace mr

extern "C" int mr_env_rollout_ddpg_collect(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                                           const mr_noise* nz, const mr_time_table* tt, const mr_rollout_io* io,
                                           const mr_ddpg_collect* c, const mr_step_out* out, void* stream) {
    mr::NvtxRange nvtx_range("mr_env_rollout_ddpg_collect");
    mr::CollectView cv;
    int rc = mr::collect_view("mr_env_rollout_ddpg_collect", st, n, dtype, p, nz, tt, io, c, out, n,
                              "more envs than the ring holds (n > capacity)", cv);
    if (rc) return rc;
    if (n == 0 || io->k_steps == 0) return MR_OK;
    const mr::Params pp = mr::to_params(*p, nz);
    const mr::TimeView tv{tt->t, tt->len};
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == MR_F64 ? mr::do_rollout<double>(*st, n, pp, nz, tv, *io, nullptr, &cv, out, s)
                           : mr::do_rollout<float>(*st, n, pp, nz, tv, *io, nullptr, &cv, out, s);
}

extern "C" int mr_env_rollout_ddpg_collect_population(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                                                      const mr_noise* nz, const mr_time_table* tt, const mr_rollout_io* io,
                                                      const mr_ddpg_collect* c, int32_t members, const mr_step_out* out,
                                                      void* stream) {
    mr::NvtxRange nvtx_range("mr_env_rollout_ddpg_collect_population");
    using mr::fail;
    const char* fn = "mr_env_rollout_ddpg_collect_population";
    if (members < 1 || members > MR_DDPG_MAX_MEMBERS) return fail(MR_ERR_ARG, "%s: members must be in 1..%d", fn, MR_DDPG_MAX_MEMBERS);
    // the tensor-core actor multiplies a whole 128-env tile by one weight matrix: a tile must not span two members
    if (n <= 0 || n % members != 0 || (n / members) % 128 != 0)
        return fail(MR_ERR_ARG, "%s: n must be members x N with N a positive multiple of 128", fn);
    mr::CollectView cv;
    int rc = mr::collect_view(fn, st, n, dtype, p, nz, tt, io, c, out, n / members,
                              "more envs per member than its ring holds (N > capacity)", cv);
    if (rc) return rc;
    cv.member_envs = n / members;
    if (io->k_steps == 0) return MR_OK;
    const mr::Params pp = mr::to_params(*p, nz);
    const mr::TimeView tv{tt->t, tt->len};
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == MR_F64 ? mr::do_rollout<double>(*st, n, pp, nz, tv, *io, nullptr, &cv, out, s)
                           : mr::do_rollout<float>(*st, n, pp, nz, tv, *io, nullptr, &cv, out, s);
}

namespace mr {
// the population evaluation through the fused rollout: no state rows, no outputs; the actors, the statistics rows, K and
// the per-member env count N are all it takes besides the task
template <class T>
static int do_evaluate(const mr_ddpg_eval& e, const Params& p, const mr_noise* nz, const TimeView& tv, int k_steps,
                       cudaStream_t s) {
    StateView<T> sv;
    memset(&sv, 0, sizeof(sv));
    RolloutView<T> rv;
    memset(&rv, 0, sizeof(rv));
    rv.actor = e.actors; rv.stats = e.stats; rv.k_steps = k_steps; rv.action_source = MR_ACTIONS_ACTOR;
    const int64_t n = (int64_t)e.members * e.member_envs;
    const OutView<T> ov = out_view<T>(nullptr, n);
    NoiseView nv = noise_view(nz, n);
    nv.offset += 1;                                   // step k at offset + 1 + k; the kernel resets at offset
    nv.table_stride = e.table_cols;
    CollectView cv;
    memset(&cv, 0, sizeof(cv));
    cv.member_envs = e.member_envs;
    EvalView<T> ev;
    ev.init = (const T*)e.init; ev.ret = e.ret; ev.length = e.length; ev.outcome = e.outcome; ev.status = e.status;
    ev.crn = e.common_random_numbers ? 1 : 0;
    switch (nz->mode) {
        case MR_NOISE_TABLE: return launch_rollout<T, MR_NOISE_TABLE>(sv, rv, ov, nv, tv, p, n, nullptr, &cv, &ev, s);
        case MR_NOISE_PHILOX: return launch_rollout<T, MR_NOISE_PHILOX>(sv, rv, ov, nv, tv, p, n, nullptr, &cv, &ev, s);
        default: return launch_rollout<T, MR_NOISE_NONE>(sv, rv, ov, nv, tv, p, n, nullptr, &cv, &ev, s);
    }
}
}  // namespace mr

extern "C" int mr_ddpg_evaluate_population(const mr_ddpg_eval* ev, int32_t dtype, const mr_sim_params* p, const mr_noise* nz,
                                           const mr_time_table* tt, void* stream) {
    mr::NvtxRange nvtx_range("mr_ddpg_evaluate_population");
    using mr::fail;
    const char* fn = "mr_ddpg_evaluate_population";
    if (!ev || !p || !nz) return fail(MR_ERR_ARG, "%s: null evaluation, params or noise", fn);
    if (!ev->actors) return fail(MR_ERR_ARG, "%s: null actor", fn);
    if (ev->members < 1 || ev->members > MR_DDPG_MAX_MEMBERS)
        return fail(MR_ERR_ARG, "%s: members must be in 1..%d", fn, MR_DDPG_MAX_MEMBERS);
    // the tensor-core actor multiplies a whole 128-env tile by one weight matrix: a tile must not span two members
    if (ev->member_envs <= 0 || ev->member_envs % 128 != 0 || ev->member_envs * ev->members > ((int64_t)1 << 31) - 1)
        return fail(MR_ERR_ARG, "%s: member_envs must be a positive multiple of 128 (and members x member_envs < 2^31)", fn);
    if (dtype != MR_F64 && dtype != MR_F32) return fail(MR_ERR_ARG, "%s: bad dtype %d", fn, dtype);
    if (p->max_timesteps < 0) return fail(MR_ERR_ARG, "%s: max_timesteps must be >= 0", fn);
    if (!(p->time_span > 0.0)) return fail(MR_ERR_ARG, "%s: time_span must be positive", fn);
    const int k_steps = p->max_timesteps + 1;         // every episode ends within the launch
    if (!tt || !tt->t || tt->len < 2 || tt->len < k_steps)
        return fail(MR_ERR_ARG, "%s: the time table must hold at least max_timesteps + 1 = %d entries", fn, k_steps);
    if (nz->offset_dev) return fail(MR_ERR_ARG, "%s: offset_dev is not supported (the step index is nz->offset)", fn);
    const int mode = nz->mode;
    if (mode != MR_NOISE_NONE && mode != MR_NOISE_TABLE && mode != MR_NOISE_PHILOX)
        return fail(MR_ERR_ARG, "%s: unknown noise mode %d", fn, mode);
    if (mode == MR_NOISE_NONE && p->noise_var != 0.0)
        return fail(MR_ERR_ARG, "%s: noise_var=%g needs a noise source (table or philox)", fn, p->noise_var);
    if (mode == MR_NOISE_TABLE) {
        if (!nz->table || nz->table_len <= 0) return fail(MR_ERR_ARG, "%s: table noise without a table (table_len <= 0)", fn);
        const int64_t cols = ev->common_random_numbers ? ev->member_envs : ev->member_envs * ev->members;
        if (ev->table_cols < cols)
            return fail(MR_ERR_ARG, "%s: the noise table has %lld columns, the evaluation reads %lld (%s)", fn,
                        (long long)ev->table_cols, (long long)cols,
                        ev->common_random_numbers ? "N with common random numbers" : "members x N");
    }
    if (mr::g_actor_path == 1)
        return fail(MR_ERR_UNSUPPORTED, "%s: the CUDA-core actor path (mr_set_actor_path(1)) has no evaluation", fn);
    mr::Params pp = mr::to_params(*p, nz);
    pp.auto_reset = 0;
    const mr::TimeView tv{tt->t, tt->len};
    cudaStream_t s = (cudaStream_t)stream;
    return dtype == MR_F64 ? mr::do_evaluate<double>(*ev, pp, nz, tv, k_steps, s)
                           : mr::do_evaluate<float>(*ev, pp, nz, tv, k_steps, s);
}
