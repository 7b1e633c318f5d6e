/*
 * mr_rl_b200 — C ABI of the B200-native rolling-microrobot environment.
 *
 * This is the drop-in boundary for the hot path of SuhailSama/MR_RL.  The reference has
 * no FFI of its own (it is pure Python); the entry points below are what a ctypes/cffi
 * binding placed behind the reference's classes would call, one per reference method:
 *
 *   mr_env_reset     <- MR_Env.reset            (MR_env.py:164-201)
 *                       Simulator.reset_start_pos (MR_simulator.py:21-34)
 *   mr_env_step      <- MR_Env.step             (MR_env.py:70-98)
 *                       Simulator.step / simulate (MR_simulator.py:36-88)
 *                       scipy RK45.__init__/_step_impl as driven from MR_simulator.py:42-50,90-91
 *                       MR_Env.convert_state / end / calculate_reward (MR_env.py:100-152)
 *   mr_env_rollout   <- utils.run_sim           (utils.py:43-61)   open-loop K-step rollout
 *                       RL/MR_ddpg.py:268-311   closed loop with ActorNetwork.predict (:124-149)
 *   mr_gp_predict    <- LearningModule.error / objective / predict -> sklearn GPR.predict
 *                       (Learning_module.py:10-24,186-224)
 *   mr_gp_correct_heading <- LearningModule.predict's minimize_scalar(objective, 'Bounded')
 *                       (Learning_module.py:215, utils.py:194-196)
 *   mr_gp_correct_action_2d <- LearningModule2D.predict's minimize over (alpha, f)  (Learning_module_2d.py:239-268)
 *   mr_actor_forward <- ActorNetwork.predict    (RL/MR_ddpg.py:124-149)
 *   mr_ddpg_update, mr_replay_add, mr_ou_noise_add <- the learner of RL/MR_ddpg.py (:16-78, :163-231, :285-305)
 *   mr_learn_preprocess <- LearningModule.estimateDisturbance / learn up to the fit (Learning_module.py:46-59, :63-120)
 *   mr_gp_fit        <- GaussianProcessRegressor.fit at given hyper-parameters: K, cholesky, alpha_, L^-1,
 *                       log marginal likelihood  (Learning_module.py:122-123; the optimiser stays on the host)
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; the library never
 *     allocates or frees caller memory and never synchronises the stream;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - functions return 0 on success, a negative mr_status on argument / launch errors and
 *     never throw; mr_last_error() gives the message for the calling thread;
 *   - per-env failures (solver failed, non-finite state, noise table exhausted) are OR-ed
 *     into the sticky per-env `status` byte instead of raising like scipy does;
 *   - `dtype` selects the STORAGE type of state/action/observation buffers (MR_F64/MR_F32);
 *     step-size control and the integrator always run in fp64 registers.
 *
 * There is no CPU fallback: every entry point launches CUDA kernels built for sm_100a.
 */
#ifndef MR_RL_B200_H
#define MR_RL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MR_ABI_VERSION 2   /* 2: per-env parameter rows, noise offset_dev, float32 I/O rows, episode recording */

enum mr_status {
    MR_OK = 0,
    MR_ERR_ARG = -1,      /* bad argument (null pointer, n < 0, misaligned buffer, ...) */
    MR_ERR_CUDA = -2,     /* kernel launch / CUDA runtime error */
    MR_ERR_UNSUPPORTED = -3
};

enum mr_dtype { MR_F64 = 0, MR_F32 = 1 };

enum mr_noise_mode {
    MR_NOISE_NONE = 0,    /* sigma == 0: no draws are consumed */
    MR_NOISE_TABLE = 1,   /* shared pre-generated standard-normal tensor (parity mode) */
    MR_NOISE_PHILOX = 2   /* counter-based in-kernel generator (throughput mode) */
};

enum mr_env_flag {        /* bits of the per-env status byte */
    MR_ENV_SOLVER_FAILED = 1,   /* scipy would return TOO_SMALL_STEP and then raise RuntimeError */
    MR_ENV_NONFINITE = 2,       /* scipy check_arguments would raise ValueError */
    MR_ENV_NOISE_OVERFLOW = 4,  /* the table noise stream of this env ran out */
    MR_ENV_ATTEMPT_CAP = 8      /* more than the attempt cap in one env step */
};

enum mr_reward_mode {
    MR_REWARD_CONST10 = 0,      /* MR_env.py:89  rew = 10 */
    MR_REWARD_SHAPED = 1        /* MR_env.py:118-134 calculate_reward (defined, unused by step) */
};

enum mr_action_source {
    MR_ACTIONS_TENSOR = 0,      /* actions[K][n][2] */
    MR_ACTIONS_PHILOX = 1,      /* uniform in action_space, generated in-kernel */
    MR_ACTIONS_ACTOR = 2,       /* DDPG actor MLP evaluated in-kernel on the observation */
    MR_ACTIONS_BROADCAST = 3    /* actions[K][2], the same action for every env (utils.run_sim) */
};

/* Simulator + env parameters (MR_simulator.py:12-19, MR_env.py:34-63).  Launch scalars. */
typedef struct mr_sim_params {
    double a0;              /* Simulator.a0 */
    double noise_var;       /* Simulator.noise_var (used as the STANDARD DEVIATION, MR_simulator.py:72) */
    int32_t is_mismatched;  /* Simulator.is_mismatched */
    int32_t mism_at_reset;  /* value of is_mismatched while reset builds the integrator
                               (MR_env.py:181 runs before :183) */
    double time_span;       /* 0.030 */
    double rtol;            /* time_span / number_iterations = 3e-4 */
    double atol;            /* 1e-4 */
    int32_t max_timesteps;  /* 50 */
    int32_t reward_mode;    /* mr_reward_mode */
    double min_dist2goal;   /* 30 */
    double bound_xy;        /* 5000  (observation_space, MR_env.py:37-39) */
    double bound_d;         /* 80000 */
    int32_t auto_reset;     /* re-initialise an env from init_space right after a terminal step (gym vector-env style) */
    int32_t action_f32;     /* != 0: the `actions` buffer of mr_env_step is float32 [n][2] although dtype is MR_F64
                               (halves the host->device bytes of a host-buffer step; the values are widened exactly) */
    double init_low[2];     /* init_space, MR_env.py:40-42 */
    double init_high[2];
    double action_high[2];  /* action_space.high, MR_env.py:34-36 */
} mr_sim_params;

/* Per-env state, structure-of-arrays: one row of n elements per field. */
typedef struct mr_env_state {
    void* x;            /* position (storage dtype) */
    void* y;
    void* fx;           /* carried derivative integrator.f (stage K0 of the next step) */
    void* fy;
    void* h;            /* carried integrator.h_abs */
    int32_t* counter;   /* MR_Env.counter == env steps since reset (t = t_table[counter]) */
    int32_t* cursor;    /* table-noise draws consumed so far (MR_NOISE_TABLE only; else may be NULL) */
    uint8_t* status;    /* sticky mr_env_flag bits */
    /* Optional per-env simulator parameters (MR_simulator.py:16-19 are per-instance attributes, set per reset at
     * MR_env.py:179-183).  All three NULL: every env uses the launch scalars of mr_sim_params.  All three given: the rows
     * are the truth for step / rollout; mr_env_reset WRITES them for the envs it resets (from its per-env new-value
     * arrays, else from the launch scalars), building the integrator with the new a0 / noise_var and the OLD flag. */
    double* a0;             /* [n] Simulator.a0 */
    double* noise_var;      /* [n] Simulator.noise_var */
    uint8_t* is_mismatched; /* [n] Simulator.is_mismatched */
} mr_env_state;

/* Per-env arguments of MR_Env.reset(noise_var, a0, is_mismatched) for mr_env_reset; any member may be NULL (= the launch
 * scalar).  Only meaningful when the state carries the per-env parameter rows. */
typedef struct mr_reset_params {
    const double* a0;             /* [n] */
    const double* noise_var;      /* [n] */
    const uint8_t* is_mismatched; /* [n] */
} mr_reset_params;

typedef struct mr_noise {
    int32_t mode;          /* mr_noise_mode */
    int32_t reserved;
    const double* table;   /* [table_len][n]: draw-major, env-minor standard normals (fp64) */
    int64_t table_len;     /* draws available per env */
    uint64_t seed;         /* Philox key */
    uint64_t offset;       /* Philox: global env-step index of this launch (caller increments) */
    uint64_t env_base;     /* global index of local env 0 (multi-GPU sharding) */
    const uint64_t* offset_dev; /* optional DEVICE counter added to `offset` when the kernel runs: launches captured in
                                   a CUDA graph keep drawing fresh noise on every replay (set it with mr_counter_set
                                   before a replay); NULL = none */
} mr_noise;

/* Inspection hook for the generated-noise mode: the first `count` standard normals of the Philox stream of env
 * env_base + i at env-step `step` — stream_id 0: the step's process noise (its first 8 values are the sufficient
 * statistics g1x, g2x, g1y, g2y of the RK45 attempt and the four draws of the rebuilt integrator, csrc/mr_core.cuh), 1: the
 * draws of an (auto) reset in that env-step — written to z_out[count][n] (float32, the generator's precision).  Lets a test
 * feed the reference's algorithm the draws the kernel used. */
int mr_philox_normals(uint64_t seed, uint64_t env_base, uint64_t step, int32_t stream_id, int32_t count, int64_t n,
                      float* z_out, void* stream);

/* *counter = value, stream-ordered (one tiny kernel): the base env-step index of the next graph replay. */
int mr_counter_set(uint64_t* counter_dev, uint64_t value, void* stream);

/* t_k after k env steps since reset, t_k = fl(t_{k-1} + time_span) (MR_simulator.py:46-50). */
typedef struct mr_time_table {
    const double* t;       /* device, [len] */
    int32_t len;
    int32_t reserved;
} mr_time_table;

typedef struct mr_step_out {
    void* obs;          /* [5][n] rows x, y, goal_x, goal_y, d (storage dtype); may be NULL */
    void* rew;          /* [n] storage dtype; may be NULL */
    uint8_t* done;      /* [n]; may be NULL */
    void* state_prime;  /* [2][n] Simulator.state_prime (MR_simulator.py:87); may be NULL */
    int64_t row_stride; /* elements between rows of obs / state_prime (0 = n) */
    int32_t skip_goal_rows; /* != 0: leave obs rows 2, 3 (the constant goal (0, 0), MR_env.py:57) untouched — the caller
                             * zeroed them once; saves 2 of the 5 obs rows when obs points at host memory */
    int32_t out_f32;        /* != 0: obs / rew / state_prime rows are float32 although dtype is MR_F64 (row_stride then
                             * counts floats): the 1e-4 tier of the outputs at half the device->host bytes, while the state
                             * and every decision stay fp64 */
} mr_step_out;

int mr_abi_version(void);
const char* mr_last_error(void);
void mr_default_params(mr_sim_params* p);

/* Tuning / test hook: force the kernel variant of mr_env_step.  0 = default choice (tiled TMA kernel, 2-D tensor maps where
 * the rows are equally strided), 1 = tiled TMA kernel with 1-D bulk copies only, 2 = 16-byte vector kernel, 3 = scalar
 * kernel, 4 = warp-specialised TMA kernel where it applies, 5 = same as 0.  Every variant computes the same
 * results (tested); returns the previous setting, or MR_ERR_ARG.  Initial value: environment variable MR_STEP_PATH
 * (tma | vec | scalar | ws).  Process-wide, not thread-safe against concurrent launches. */
int mr_set_step_path(int32_t path);

/* The same for the actor evaluated inside mr_env_rollout (MR_ACTIONS_ACTOR): 0 = default (both dense layers on the
 * tensor cores, 3xFP16 passes, four CTAs per SM), 1 = CUDA-core MLP, 2 = hidden layer on the tensor cores with 3xTF32
 * passes (fp32 operand range).  Initial value: environment variable MR_ACTOR_PATH (simt | tf32).  Returns the previous one. */
int mr_set_actor_path(int32_t path);

/* Fill t[0..len) on the HOST with the accumulated step times. */
void mr_fill_time_table_host(double* t_host, int32_t len, double time_span);

/*
 * MR_Env.reset for every env with mask[i] != 0 (mask == NULL: all).  init_xy is [n][2]
 * (storage dtype) or NULL to sample init_space with Philox (float32-rounded like
 * gym.spaces.Box.sample).  reset_cursor != 0 rewinds the table-noise cursor to 0.
 */
int mr_env_reset(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                 const mr_noise* nz, const void* init_xy, const uint8_t* mask, int32_t reset_cursor,
                 const mr_step_out* out, void* stream);
/* The same with per-env reset arguments (rp may be NULL = mr_env_reset). */
int mr_env_reset_ex(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                    const mr_noise* nz, const void* init_xy, const uint8_t* mask, int32_t reset_cursor,
                    const mr_reset_params* rp, const mr_step_out* out, void* stream);

/* MR_Env.step for n envs.  actions is [n][2] (f_t, alpha_t), storage dtype. */
/* (device buffers; the host-buffer form is mr_env_step_host below) */
int mr_env_step(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                const mr_noise* nz, const mr_time_table* tt, const void* actions,
                const mr_step_out* out, void* stream);

typedef struct mr_rollout_io {
    int32_t action_source;   /* mr_action_source */
    int32_t k_steps;         /* env steps fused in this launch, state held in registers */
    const void* actions;     /* TENSOR: [K][n][2]; BROADCAST: [K][2]; storage dtype */
    const float* actor;      /* ACTOR: packed weights, see mr_actor_param_count() */
    void* traj_xy;           /* optional [K][2][n] positions after each step (run_sim X, Y) */
    void* traj_state_prime;  /* optional [K][2][n] */
    uint8_t* traj_done;      /* optional [K][n] */
    double* stats;           /* optional [MR_STATS_LEN] device accumulators (atomically added) */
    /* Per-episode recording on the device — what MRExperiment.new_iter / new_transition log (MR_data.py:27-57,
     * MR_env.py:94-95,190-198) — all optional, storage dtype unless noted: */
    void* traj_actions;      /* [K][n][2] the action applied at step k (also for the in-kernel policies) */
    void* traj_rew;          /* [K][n] reward of step k */
    void* traj_reset_xy;     /* [K][2][n] written where traj_done[k][i] != 0 and auto_reset is on: the start position of
                                the episode that follows (row 0 of the next iteration's log) */
    int32_t* traj_episode;   /* [K][n] ordinal of the episode of env i the transition belongs to */
    int32_t* traj_step;      /* [K][n] step inside that episode (MR_Env.counter after the step) */
    int32_t* episode_counter;/* [n] in/out: episodes env i has finished so far (carries the ordinals across launches) */
    const void* reset_init;  /* [reset_init_len][n][2] start positions of the auto resets: the e-th finished episode of
                                env i is followed by reset_init[(e - 1) % reset_init_len][i]; NULL: sample init_space
                                (gym Box.sample, MR_env.py:172-173) */
    int32_t reset_init_len;
    int32_t reserved;
} mr_rollout_io;

enum { MR_STAT_EPISODES = 0, MR_STAT_SUM_LENGTH = 1, MR_STAT_SUM_REWARD = 2, MR_STAT_GOAL = 3,
       MR_STAT_OUT_OF_BOUNDS = 4, MR_STAT_TIMEOUT = 5, MR_STAT_ENV_STEPS = 6, MR_STAT_FAILED = 7,
       MR_STATS_LEN = 8 };

/* K fused MR_Env.step calls (utils.run_sim / the DDPG acting loop).  `out` receives the
 * outputs of the LAST step. */
int mr_env_rollout(const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                   const mr_noise* nz, const mr_time_table* tt, const mr_rollout_io* io,
                   const mr_step_out* out, void* stream);

/* ---- Gaussian-process inference (Learning_module.py -> sklearn GPR.predict) ----------
 * The fitted model (GPR.X_train_, alpha_, L_, kernel_ = RBF(length_scale) + WhiteKernel(noise_level))
 * is prepared once on the host: arrays are zero-padded from n_train to n_pad (a multiple of
 * MR_GP_PAD) so the tiled kernels need no bounds checks.  Padded training points carry
 * alpha = 0 and zero rows/columns of linv, so they contribute nothing. */
#define MR_GP_PAD 128

typedef struct mr_gp_model {
    const double* x_train_scaled; /* [n_pad][dim]  GPR.X_train_ / length_scale (sklearn RBF scales first) */
    const double* alpha;     /* [n_pad]  GPR.alpha_ (0 in the padding) */
    const double* linv;      /* proj_rows == 0: [n_pad][n_pad] row-major inverse of the lower Cholesky factor GPR.L_,
                                upper triangle and padding zero.  proj_rows > 0: [proj_rows][n_pad] dense spectral
                                projection P with |P k|^2 = k^T K^-1 k (rows u_i^T / sqrt(mu_i) of the leading
                                eigenpairs of K; the RBF Gram matrix is numerically low rank, so a few hundred rows
                                reproduce the triangular form to rounding at a fraction of its cost).
                                NULL if std is never requested */
    int32_t n_train;
    int32_t n_pad;
    int32_t dim;             /* 1 (Learning_module.py) or 2 (Learning_module_2d.py) */
    int32_t proj_rows;       /* 0, or the number of projection rows: 32, 64, 96 or a multiple of MR_GP_PAD */
    double length_scale;     /* kernel_.k1.length_scale */
    double noise_level;      /* kernel_.k2.noise_level */
} mr_gp_model;

/* mean[i] = k(q_i, X) . alpha ;  std[i] = sqrt(max(0, 1 + noise_level - |linv k(q_i, X)|^2)).
 * q is [n_q][dim].  std may be NULL (mean only, Learning_module.py:17-18,207-208); then no
 * workspace is needed.  workspace must hold mr_gp_workspace_bytes() bytes. */
int mr_gp_predict(const mr_gp_model* gp, const double* q, int64_t n_q, double* mean, double* std,
                  void* workspace, int64_t workspace_bytes, void* stream);
int64_t mr_gp_workspace_bytes(const mr_gp_model* gp, int64_t n_q, int32_t want_std);

/* LearningModule.predict's search (Learning_module.py:198-215, utils.find_alpha_corrected) for n desired
 * velocities vd[n][2]: bounded scalar minimisation over alpha in [-pi, pi] (scipy _minimize_scalar_bounded:
 * golden section + parabolic steps, xatol 1e-5, maxiter 500) of `objective` (Learning_module.py:10-24) with
 * both GP means evaluated on the device inside the loop.  alpha_out[n]; nfev_out[n] may be NULL.  The
 * posterior at the minimiser (Learning_module.py:221-222) is a following mr_gp_predict call. */
int mr_gp_correct_heading(const mr_gp_model* gpx, const mr_gp_model* gpy, const double* vd, int64_t n, double a0,
                          double freq, double drift_x, double drift_y, double* alpha_out, int32_t* nfev_out, void* stream);

/* GaussianProcessRegressor.fit for kernel RBF(length_scale) + WhiteKernel(noise_level) at FIXED hyper-parameters
 * (Learning_module.py:30-33,122-123): K = rbf(X/l) + (noise_level + jitter) I  (jitter = sklearn's alpha, 1e-10),
 * L = chol(K), alpha = K^-1 y, linv = L^-1, lml = -0.5 y.alpha - sum log L_ii - n/2 log 2pi.
 * x_train [n_train][dim], y [n_train].  Outputs are laid out as mr_gp_model wants them: x_scaled_out
 * [n_pad][dim], alpha_out [n_pad], linv_out [n_pad][n_pad] (padding zero); lml_out (1 double), grad_out
 * (2 doubles: d lml / d log length_scale, d lml / d log noise_level — what sklearn's optimiser consumes) and
 * info_out (1 int32: 0, or 1 + the first non-positive pivot like LAPACK potrf) may be NULL.  n_pad must be a multiple of
 * MR_GP_PAD; workspace must hold mr_gp_fit_workspace_bytes(n_pad) bytes, 16-byte aligned. */
int mr_gp_fit(const double* x_train, const double* y, int32_t n_train, int32_t n_pad, int32_t dim, double length_scale,
              double noise_level, double jitter, double* x_scaled_out, double* alpha_out, double* linv_out,
              double* lml_out, double* grad_out, int32_t* info_out, void* workspace, int64_t workspace_bytes, void* stream);
int64_t mr_gp_fit_workspace_bytes(int32_t n_pad);

/* mr_gp_correct_heading with the two GP means given as Chebyshev series on the search interval [-pi, pi]
 * (mu(alpha) = sum_k coef[k] T_k(alpha / pi)): a GP mean with an RBF kernel is an entire function of the heading, so a
 * few hundred coefficients carry it to the accuracy of the direct sum and one evaluation is a Clenshaw pass instead of
 * 2 x n_train exponentials.  The caller samples the means with mr_gp_predict, builds the series and CHECKS them against
 * mr_gp_predict before relying on this entry point (mr_rl_b200/learning_module.py does).  Same search, same outputs. */
int mr_gp_correct_heading_cheb(const double* coef_x, const double* coef_y, int32_t n_coef, const double* vd, int64_t n,
                               double a0, double freq, double drift_x, double drift_y, double* alpha_out, int32_t* nfev_out,
                               void* stream);

/* LearningModule2D.predict's search (Learning_module_2d.py:239-268) for n desired velocities vd[n][2]: the minimiser over
 * (alpha, f) in the box [lo, hi] of |a0 f (cos alpha, sin alpha) + (muX, muY)(alpha, f) - vd|^2 (= the reference's objective),
 * both GP means and their gradients evaluated on the device, started at clip((atan2(vd), |vd| / a0)).  x_out[n][2];
 * iters_out[n] (passes used) and status_out[n] (0 converged, 1 pass cap, 2 non-finite) may be NULL.  The posterior at the
 * minimiser is a following mr_gp_predict call.  lo, hi, a0 are host values; gpx, gpy must be dim-2 models over the same
 * training inputs.  The search is a projected Newton / Levenberg-Marquardt method on the box (csrc/mr_gp.cu), not a port
 * of scipy's L-BFGS-B; where the minimum is unique the two end at the same point to within L-BFGS-B's own tolerance. */
int mr_gp_correct_action_2d(const mr_gp_model* gpx, const mr_gp_model* gpy, const double* vd, int64_t n, double a0,
                            const double lo[2], const double hi[2], double* x_out, int32_t* iters_out, uint8_t* status_out,
                            void* stream);

/* ---- DDPG actor forward (RL/MR_ddpg.py:124-149) --------------------------------------
 * Packed float32 parameters (input-major matrices W[in][out]):
 *   w1[5][64] b1[64] gamma1[64] beta1[64] mean1[64] var1[64]
 *   w2[64][64] b2[64] gamma2[64] beta2[64] mean2[64] var2[64]   w3[64][2] b3[2]          */
int32_t mr_actor_param_count(void);
/* obs is [5][obs_row_stride] (storage dtype), actions out is [n][2] (storage dtype). */
int mr_actor_forward(const float* actor, const void* obs, int64_t obs_row_stride, int64_t n, int32_t dtype,
                     const double action_high[2], void* actions, void* stream);

/* ---- MR_Env.step with HOST buffers (what a caller holding numpy arrays does per control step, MR_env.py:70-98) ----
 * Unlike every other entry point this one BLOCKS until the host buffers are filled.  Two strategies:
 *   n_chunks == 0  DIRECT: the step kernel reads the actions from and writes obs / reward / done to the host buffers
 *                  itself (one launch; its bulk copies cross PCIe in both directions while the state stays in HBM).
 *                  The host buffers must be page-locked and device-addressable (cudaHostAlloc / cudaHostRegister under
 *                  unified addressing, e.g. torch pinned memory), rows 16-byte aligned.  pl, actions_dev, out_dev may be
 *                  NULL (out_dev->state_prime, if given, is still written on the device).  This is the fast path.
 *   n_chunks >= 1  STAGED: H2D of the actions, the step kernel and D2H of the results, split into env ranges pipelined
 *                  on three internal streams (copy-in of chunk i+1, kernel of chunk i, copy-out of chunk i-1 overlap).
 *                  Works with any page-locked host memory (with io->actions_dev == NULL the chunk kernels read the
 *                  actions from the host buffer themselves, which then has to be device-addressable as in the direct
 *                  mode).  The x, y rows go out as one 2-D copy per chunk.  The pipeline object owns only CUDA streams
 *                  and events.  Measured at 2^20 envs: direct 0.66-0.68 ms, staged 0.73 ms (2 chunks). */
typedef struct mr_host_pipeline mr_host_pipeline;
int mr_host_pipeline_create(int32_t max_chunks, mr_host_pipeline** out);
void mr_host_pipeline_destroy(mr_host_pipeline* pl);

typedef struct mr_host_step_io {
    const void* actions_host;  /* HOST  [n][2] (f_t, alpha_t), storage dtype                                  */
    void* actions_dev;         /* device staging [n][2] (staged mode; NULL = the chunk kernels read            */
                               /*       actions_host themselves and only the results use the copy engine)     */
    void* obs_host;            /* HOST  [5][host_row_stride]; rows 2, 3 (the constant goal) are copied only if  */
    void* rew_host;            /* HOST  [n]                                     copy_goal_rows != 0           */
                               /*       (may be NULL — with the constant reward of MR_env.py:89 there is      */
                               /*        nothing to send)                                                     */
    uint8_t* done_host;        /* HOST  [n]                                                                   */
    int64_t host_row_stride;   /* elements between obs_host rows (0 = n)                                      */
    int32_t copy_goal_rows;
    int32_t io_f32;            /* direct mode, MR_F64 storage: actions_host / obs_host / rew_host are float32 */
                               /* (the 1e-4 tier on the wire; the state and all decisions stay fp64)          */
} mr_host_step_io;

/* Page-lock a caller-owned host range in place (cudaHostRegister) so the direct mode can read / write it without a
 * staging copy — for callers that step with the same plain (malloc'ed, numpy) buffers every time.  Fails with
 * MR_ERR_UNSUPPORTED where registered memory is not addressable by its host pointer.  Undo with mr_host_unregister
 * before the memory is freed. */
int mr_host_register(void* host_ptr, int64_t bytes);
int mr_host_unregister(void* host_ptr);

/* out_dev: the device rows the kernel writes (obs, rew, done required).  `stream`: the caller's stream; the pipeline
 * starts after the work already queued on it, and work queued on it afterwards sees the stepped state. */
int mr_env_step_host(mr_host_pipeline* pl, const mr_env_state* st, int64_t n, int32_t dtype, const mr_sim_params* p,
                     const mr_noise* nz, const mr_time_table* tt, const mr_host_step_io* io, const mr_step_out* out_dev,
                     int32_t n_chunks, void* stream);

/* LearningModule.estimateDisturbance / learn up to the GPR fit (Learning_module.py:46-59, :63-120) for a trajectory
 * px, py, time [n] already in HBM: uniform_filter1d(N, nearest) -> np.gradient(., time) -> uniform_filter1d(N/2)
 * gives vx_out, vy_out [n]; scalars_out[0..1] = mean of vx, vy over [N, n-N) (the drift estimate Dx, Dy).
 * With alpha_sim != NULL (learn): frames [N, n_valid-N) of the controller-on part (n_valid = n, or the cut the caller
 * derived from alpha >= 500) give a0 = median(speed / freq) -> scalars_out[2], the sample count m -> scalars_out[3],
 * x_out = alpha_sim, yx_out / yy_out = vx - a0 freq cos(alpha) / vy - a0 freq sin(alpha), m entries each — the
 * inputs of mr_gp_fit.  subtract_t0 shifts the clock like learn() does (:70).  workspace: mr_learn_workspace_bytes(n). */
int mr_learn_preprocess(const double* px, const double* py, const double* time, int32_t n, int32_t filter_n, int32_t subtract_t0,
                        double drift_x, double drift_y, const double* alpha_sim, double freq, int32_t n_valid, double* vx_out,
                        double* vy_out, double* x_out, double* yx_out, double* yy_out, double* scalars_out, void* workspace,
                        int64_t workspace_bytes, void* stream);
int64_t mr_learn_workspace_bytes(int32_t n);

/* ---- DDPG learner (RL/MR_ddpg.py:16-78,80-231,285-305; SURVEY §8f rank 3) ---------------------------
 * Packed float32 critic parameters (input-major matrices), mr_critic_param_count() floats:
 *   wc1[5][64] bc1[64] gamma[64] beta[64] mean[64] var[64]  t1[64][32] t1b[32] (unused, as in the reference)
 *   t2[2][32] t2b[32]  wo[32] bo[1]
 * The learner state is eight parameter-sized device arrays plus two gradient scratch arrays; the replay ring is
 * five row-major float32 arrays of `capacity` rows.  The caller owns head / count / Adam's step number. */
typedef struct mr_ddpg_state {
    float* actor;          /* [mr_actor_param_count()]  online actor  (ActorNetwork.network_params)        */
    float* actor_target;   /*                            target actor  (:93-103)                             */
    float* critic;         /* [mr_critic_param_count()] online critic (CriticNetwork.network_params)       */
    float* critic_target;
    float* adam_actor_m;   /* Adam first / second moments, same layouts                                      */
    float* adam_actor_v;
    float* adam_critic_m;
    float* adam_critic_v;
    float* grad_actor;     /* scratch, same layouts                                                          */
    float* grad_critic;
} mr_ddpg_state;

typedef struct mr_replay {
    float* s;              /* [capacity][5]  state                    (ReplayBuffer.add, :27-35)            */
    float* a;              /* [capacity][2]  action                                                          */
    float* r;              /* [capacity]     reward                                                          */
    float* d;              /* [capacity]     terminal flag as 0 / 1                                          */
    float* s2;             /* [capacity][5]  next state                                                      */
    int64_t capacity;
} mr_replay;

typedef struct mr_ddpg_hyper {
    double gamma, tau, lr_actor, lr_critic;     /* 0.99, 0.001, 0.001, 0.01   (RL/MR_ddpg.py:337-341)        */
    double action_bound[2];                      /* env.action_space.high                                     */
    double adam_beta1, adam_beta2, adam_eps;     /* TF1 AdamOptimizer defaults 0.9, 0.999, 1e-8               */
} mr_ddpg_hyper;

int32_t mr_critic_param_count(void);

/* ReplayBuffer.add for the n transitions of one vectorised env step: transition i goes to ring slot
 * (head + i) % capacity.  obs / obs_next are SoA rows [5][row_stride], actions [n][2], rew [n] (storage dtype),
 * done [n] bytes.  The caller advances head by n (mod capacity) and count to min(count + n, capacity). */
int mr_replay_add(const mr_replay* rb, int64_t head, const void* obs, int64_t obs_row_stride, const void* actions,
                  const void* rew, const uint8_t* done, const void* obs_next, int64_t obs_next_row_stride, int64_t n,
                  int32_t dtype, void* stream);

/* OUNoise.__call__ (:67-71) for n envs: ou_state [n][2] float64 is advanced by one step with Philox normals keyed by
 * (seed; env_base + i, counter) and added to actions [n][2] in place; envs with reset_mask[i] != 0 (may be NULL)
 * restart from 0 first (OUNoise.reset). */
int mr_ou_noise_add(double* ou_state, void* actions, const uint8_t* reset_mask, int64_t n, int32_t dtype, double theta, double mu,
                    double sigma, double dt, uint64_t seed, uint64_t counter, uint64_t env_base, void* stream);

/* One pass of the reference's update block (:285-305) in ONE launch: minibatch (rows `indices[batch]`, or if NULL a
 * uniform sample without replacement from the first `count` ring rows, Philox keyed by (seed; update_index)),
 * y = r + gamma Q'(s2, mu'(s2)) (1 - done), critic MSE step (Adam), dQ/da at mu(s) under the updated critic, actor
 * step (Adam on d scaled_out/d theta . (-dQ/da) / batch), soft target updates.  update_index = 1, 2, ... is Adam's
 * step count.  info_out (2 floats, may be NULL): critic loss and mean Q before the update. */
int mr_ddpg_update(const mr_ddpg_state* st, const mr_replay* rb, int64_t count, int32_t batch, const int64_t* indices,
                   uint64_t seed, int64_t update_index, const mr_ddpg_hyper* hp, float* info_out, void* workspace,
                   int64_t workspace_bytes, void* stream);
/* Minibatches above 64 samples run data-parallel over one CTA per SM (four launches: critic gradients, critic Adam,
 * actor gradients, actor Adam; per-CTA partial gradients summed in a fixed order) when a workspace of
 * mr_ddpg_workspace_bytes(batch) bytes is passed; without one (NULL) the single-CTA kernel handles up to 4096 samples.
 * Sampling in that path is mr_replay_sample's. */
int64_t mr_ddpg_workspace_bytes(int32_t batch);

/* The two halves of the data-parallel update as separate steps, for learners that exchange gradients between ranks
 * (one process per GPU, each with its own replay shard): mr_ddpg_gradients leaves the summed gradient of this rank's
 * minibatch in grad_out — which = 0: critic, mr_critic_param_count() + 2 floats (the last two: the sums of the squared TD errors
 * and of Q over the minibatch); which = 1: actor, mr_actor_param_count() floats, through the CURRENT
 * critic — the caller all-reduces it (NCCL) and hands it to mr_ddpg_apply with grad_scale = 1 / world_size, which does
 * Adam and the soft target update.  Order per update: gradients(0), apply(0), gradients(1), apply(1); both gradient
 * calls of one update see the same rows (given, or regenerated from (seed, update_index)). */
int mr_ddpg_gradients(const mr_ddpg_state* st, const mr_replay* rb, int64_t count, int32_t batch, const int64_t* indices,
                      uint64_t seed, int64_t update_index, const mr_ddpg_hyper* hp, int32_t which, float* grad_out,
                      void* workspace, int64_t workspace_bytes, void* stream);
int mr_ddpg_apply(const mr_ddpg_state* st, int32_t which, const float* grad, double grad_scale, int64_t update_index,
                  const mr_ddpg_hyper* hp, void* stream);

/* `batch` distinct ring rows out of the first `count`, uniformly at random (random.sample, RL/MR_ddpg.py:43-46), in
 * parallel: a keyed bijection (4-round Feistel network, keys from Philox(seed; update_index)) of a power-of-four domain
 * cycle-walked into [0, count).  indices_out: device int64 [batch]. */
int mr_replay_sample(int64_t count, int32_t batch, uint64_t seed, int64_t update_index, int64_t* indices_out, void* stream);

/* mr_actor_forward for MR_Env observations — obs rows 2, 3 (the goal) are identically zero (MR_env.py:57) and are not
 * read — with the hidden layer on the tensor cores (tcgen05, 3xTF32 ~ fp32 accuracy).  Same arguments. */
int mr_actor_forward_env(const float* actor, const void* obs, int64_t obs_row_stride, int64_t n, int32_t dtype,
                         const double action_high[2], void* actions, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MR_RL_B200_H */
