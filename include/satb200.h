/*
 * satb200.h -- C ABI of libsatb200.so: the B200 (sm_100a) implementation of the batched satellite
 * environment step of qiaobeibei/PPO-RL-Satellite.
 *
 * The reference has no FFI boundary (it is in-process Python); this header is the boundary the
 * drop-in defines (SURVEY.md s8b tier 2). Each entry point cites the reference interface it
 * replaces (file:line relative to the upstream repository). The Python facade in
 * ppo-rl-satellite_b200/ binds these symbols with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in _host;
 *     the library never allocates on behalf of the caller and keeps no global state
 *   - every call enqueues on `stream` (a cudaStream_t passed as void*) and returns immediately;
 *     *_host entry points copy in, run, copy out and synchronise the stream before returning
 *   - return value: 0 ok; <0 argument error (SAT_ERR_*); >0 the cudaError_t of the launch
 *   - SoA columns are 16-byte aligned and `ld` (column stride, in elements) is a multiple of 2
 *   - thread-safe and re-entrant; one CUDA context per process/GPU is the expected use
 */
#ifndef SATB200_H
#define SATB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SATB200_ABI_VERSION 3

#define SAT_OK          0
#define SAT_ERR_NULL   -1   /* required pointer is NULL */
#define SAT_ERR_SIZE   -2   /* bad size / stride / alignment */
#define SAT_ERR_MODE   -3   /* bad enum value */

int         sat_abi_version(void);
const char* sat_strerror(int code);          /* static strings; >0 codes map to cudaGetErrorString */

/* ------------------------------------------------------------------------------------------------
 * K1  RK4 two-body(+J2) propagator.
 * Replaces StateEq + RungeKutta ("轨道外推-龙格库塔算法.py":15-40) applied `substeps` times with step h
 * to n independent states. x is SoA [6][ld]: rows x,y,z,vx,vy,vz. j2 = 0 gives pure two-body.
 * Units are the caller's (km: mu=398600, re=6378.137; m: mu=3.986e14, re=6378137).
 * ------------------------------------------------------------------------------------------------ */
int sat_rk4_propagate(double* x, int64_t n, int64_t ld, double h, int substeps,
                      double mu, double re, double j2, void* stream);
/* host-buffer form: x_host is [6][n] in pageable or pinned host memory; d_scratch is a device
 * buffer of 6*ld doubles provided by the caller (ld >= n, even). */
int sat_rk4_propagate_host(double* x_host, int64_t n, double* d_scratch, int64_t ld, double h,
                           int substeps, double mu, double re, double j2, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2  fused environment step.
 * Replaces satellites.reset / satellites.step (environment.py:66-79, 81-255) for n independent envs,
 * including Clohessy_Wiltshire.State_transition_matrix (satellite_function.py:753-781),
 * calculate_number_hanger_area (environment.py:317-332 -> satellite_function.py:18-99,161-255,
 * 317-373,462-565 incl. scipy fsolve) and reward_of_action1-4 (environment.py:346-396).
 * ------------------------------------------------------------------------------------------------ */
enum { SAT_COL_P = 0, SAT_COL_PV = 3, SAT_COL_E = 6, SAT_COL_EV = 9,
       SAT_COL_FUEL_C = 12, SAT_COL_FUEL_T = 13, SAT_COL_DIS = 14, SAT_COL_RET = 15, SAT_STATE_COLS = 16 };
enum { SAT_ICOL_DZ = 0, SAT_ICOL_COUNT = 1, SAT_ICOL_INTSTATE = 2, SAT_ICOL_ERR = 3, SAT_ISTATE_COLS = 4 };

typedef struct {
    double*  state;    /* [SAT_STATE_COLS][ld] fp64: P(3) Pv(3) E(3) Ev(3) fuel_c fuel_t dis R(discounted return);
                        * [SAT_STATE_COLS_STARTS][ld] with the per-env start columns (below) */
    int32_t* istate;   /* [SAT_ISTATE_COLS][ld]: dangerous_zone, episode step count, int_state (Q1), err */
    int64_t  n;        /* number of environments */
    int64_t  ld;       /* column stride (elements), >= n, even */
} SatEnvState;

enum { SAT_MODE_CW = 0, SAT_MODE_RK4 = 1 };
enum { SAT_ACT_F32 = 0, SAT_ACT_F64 = 1 };

typedef struct {
    int32_t mode;               /* SAT_MODE_CW: the shipped env (CW STM); SAT_MODE_RK4: S RK4 substeps (inertial) */
    int32_t flag;               /* 0 pursuer training (environment.py:83-179), 1 evader training (:181-255) */
    int32_t max_episode_steps;  /* environment.py:46 */
    int32_t auto_reset;         /* 0: none; SAT_RESET_STARTS (2): envs that finish are reset to their start columns in the
                                 * same launch (needs a SAT_STATE_COLS_STARTS-column state buffer); any other non-zero
                                 * value: reset to reset_p / reset_e in the same launch (batched contract) */
    int32_t action_dtype;       /* SAT_ACT_F32 / SAT_ACT_F64; layout [n][3] */
    int32_t substeps;           /* rk4 mode: RK4 substeps per env step */
    int32_t skip_danger_zone;   /* 1: do not evaluate the danger-zone count (keeps it at its stale value) */
    int32_t fast_libm;          /* 0 (default): the danger-zone path performs the host libm's own arithmetic (csrc/glibm.cuh),
                                 * the integer count is the reference's bit for bit; 1: CUDA libdevice + x*x (1-2 ulp from the
                                 * host libm: ~3e-5 of the counts differ), 24 us faster per 65 536-env step */
    double  d_capture, d_range; /* environment.py:35,45 */
    double  gamma;              /* reward-scaling discount (normalization.py:57) */
    double  stm[36];            /* cw mode: row-major 6x6 STM for one step (satellite_function.py:766-773) */
    double  h, mu, re, j2;      /* rk4 mode: substep size and gravity constants (metres) */
    double  r_cw[3], v_cw[3];   /* relative->inertial translation (environment.py:338-339) */
    double  u_grav;             /* danger-zone gravitational parameter (satellite_function.py:28) */
    double  reset_p[3], reset_e[3]; /* reset() initial positions (environment.py:67,70); velocities are 0 */
} SatEnvParams;

/* running statistics block (RunningMeanStd, normalization.py:7-29), device resident:
 * [0] = n, [1..dim] = mean, [1+dim..2dim] = S, [1+2dim..3dim] = std  -> 1 + 3*dim doubles */
#define SAT_STATS_DOUBLES(dim) (1 + 3 * (dim))

/* bytes of caller-provided workspace sat_env_step / sat_norm_update need for n rows */
int64_t sat_workspace_bytes(int64_t n);

void sat_env_default_params(SatEnvParams* p);     /* reference literals; cw STM left zero */

/* constructor state (environment.py:41-44: fuel 320/320, dis=inf, dangerous_zone=0) followed by reset() */
int sat_env_init(const SatEnvState* st, double fuel_c, double fuel_t, const SatEnvParams* p, void* stream);
/* reset(Flag) (environment.py:66-79) for envs whose mask byte is non-zero (mask NULL = all).
 * fuel / dis / dangerous_zone persist exactly as in the reference (they are never reset there). */
int sat_env_reset(const SatEnvState* st, const uint8_t* mask, const SatEnvParams* p, void* stream);
/* Per-env start states. A state buffer of SAT_STATE_COLS_STARTS columns holds in columns SAT_COL_START .. +11 each env's
 * NEXT start, in the order of columns 0..11 (P, Pv, E, Ev, CW frame, metres and m/s). With auto_reset == SAT_RESET_STARTS,
 * sat_env_step / sat_env_step_timed / sat_env_step_host reset a finished env to its start columns: kinematics from the
 * columns, count = 0 and int_state = 0 (a float start has no int64 truncation, Q1); fuel, dis, dangerous_zone persist and
 * the discounted return resets on done, as in the default reset. The step does not redraw the starts: call
 * sat_env_draw_starts with the step's done mask afterwards. The columns are ordinary device memory: a caller who wants
 * another distribution writes them directly. */
enum { SAT_COL_START = 16, SAT_STATE_COLS_STARTS = 28 };
#define SAT_RESET_STARTS 2
/* draw the next start of every env whose mask byte is non-zero (mask NULL = all) into the start columns, uniform in the
 * box lo_host[c] <= x <= hi_host[c] (lo == hi fixes a column). lo_host / hi_host: [12] host arrays copied into the launch.
 * Keyed by (seed, row_offset + env index, draw) only: Philox4x32-10, key (uint32)seed, (uint32)(seed >> 32) ^ 0x53434E31,
 * counter (g_lo, g_hi, draw, j) for j = 0..5; block j's (c0, c1) and (c2, c3) give columns 2j and 2j + 1 as
 * u = ((c_a << 32 | c_b) >> 11) * 2^-53 and x = min(lo + (hi - lo) * u, hi), each operation rounded, x = lo when lo == hi.
 * NULL bounds: SAT_ERR_NULL; lo > hi, a non-finite bound or box width, row_offset < 0: SAT_ERR_SIZE. */
int sat_env_draw_starts(const SatEnvState* st, const uint8_t* mask, const double* lo_host, const double* hi_host,
                        uint64_t seed, uint32_t draw, int64_t row_offset, void* stream);
/* reset() to the start columns for the masked envs (mask NULL = all): kinematics, count = 0, int_state = 0 */
int sat_env_reset_starts(const SatEnvState* st, const uint8_t* mask, void* stream);
/* observation of the current state: [n][18] = [P-E, Pv-Ev, P, Pv, E, Ev] (environment.py:76-77) */
int sat_env_observe(const SatEnvState* st, float* obs_f32, double* obs_f64, void* stream);
/* The fp32 observation the policy networks are fed: rebuilt from the fp64 state (environment.py:76-77) and, when obs_stats !=
 * NULL, normalised in fp64 with (x - mean)/(std + 1e-8) (Normalization.__call__ with update=False, normalization.py:37-43)
 * before the cast - the arithmetic of sat_actor_sample's fused path, as one streaming kernel. */
int sat_env_observe_norm(const SatEnvState* st, const double* obs_stats, float* obs_f32, void* stream);

/* one step() for all envs.
 *   pa, ea          [n][3] pursuer / escaper actions (dtype per params)
 *   count_override  nullable [n]: the `epsiode_count` argument of step(); NULL = internal counter + 1
 *   obs_f32/obs_f64 nullable [n][18]: next observation (after auto-reset when enabled)
 *   term_obs_f64    nullable [n][18]: observation before auto-reset (the reference's returned s_)
 *   reward [n] fp64, done [n] u8: as returned by the reference
 *   obs_stats / ret_stats  nullable running statistics (dim 18 / dim 1) updated with this step's
 *                   observations / discounted returns (Normalization, RewardScaling); ret_std_out
 *                   nullable scalar that receives std(R) after the update
 *   workspace       sat_workspace_bytes(n) bytes, only needed when a stats pointer is given */
int sat_env_step(const SatEnvState* st, const void* pa, const void* ea, const int32_t* count_override,
                 float* obs_f32, double* obs_f64, double* term_obs_f64, double* reward, uint8_t* done,
                 double* obs_stats, double* ret_stats, double* ret_std_out, void* workspace,
                 const SatEnvParams* p, void* stream);

/* Measurement form of sat_env_step (bench.py): the same launches with CUDA events recorded between them on `stream`;
 * synchronises, then ms_out[0..2] (host) = front (propagation) kernel, finish kernel, statistics merge. In cw mode the
 * single fused kernel is reported in ms_out[1] and ms_out[0] is ~0. */
int sat_env_step_timed(const SatEnvState* st, const void* pa, const void* ea, const int32_t* count_override,
                       float* obs_f32, double* obs_f64, double* term_obs_f64, double* reward, uint8_t* done,
                       double* obs_stats, double* ret_stats, double* ret_std_out, void* workspace,
                       const SatEnvParams* p, void* stream, float* ms_out);

/* batched danger-zone count on explicit inertial states. Replaces
 * Time_window_of_danger_zone(R0_c, V0_c, R0_t, V0_t, Delta_V_c).calculate_number_of_hanger_area()
 * (satellite_function.py:18-99, 341-373). rv [n][12] = R0_c, V0_c, R0_t, V0_t; dv [n] = Delta_V_c.
 * count_out [n]: 0/1/2, or -1 where the reference would raise (circular / parabolic element set).
 * debug_out (nullable) [n][2][8]: per node rf_max, rf_min, r_ft, alpha(+pi/2), alpha(-pi/2), theta, dVm, f_c. */
int sat_danger_zone_count(const double* rv, const double* dv, int64_t n, double u_grav, int32_t* count_out,
                          double* debug_out, void* stream);

/* batched Numerical_iteration_method(u, Delta_Vm, theta, v_1x, v_1y, h, alpha_guess) (satellite_function.py:558-565):
 * one scipy.optimize.fsolve (MINPACK hybrd, n = 1) root of P_fai_equation per element, returned un-polished like the
 * reference's result[0]. All arrays [n] fp64 on the device; nfev_out (nullable) [n] int32 = function evaluations. */
int sat_fsolve_pfai(const double* dvm, const double* theta, const double* v1x, const double* v1y, const double* h,
                    const double* guess, int64_t n, double u_grav, double* root_out, int32_t* nfev_out, void* stream);

/* elementwise evaluation of the device libm the danger-zone path uses (csrc/glibm.cuh), so tests can compare it bit for
 * bit with the host libm the reference calls: fn = SAT_LIBM_SIN / COS / ACOS / ATAN / POW2 (numpy scalar sin, cos,
 * arccos, arctan and python `x ** 2`), SINCOS_S / SINCOS_C = the fused form's two outputs. x, y [n] fp64 on the device. */
#define SAT_LIBM_SIN 0
#define SAT_LIBM_COS 1
#define SAT_LIBM_ACOS 2
#define SAT_LIBM_ATAN 3
#define SAT_LIBM_POW2 4
#define SAT_LIBM_SINCOS_S 5
#define SAT_LIBM_SINCOS_C 6
int sat_libm_eval(int fn, const double* x, double* y, int64_t n, void* stream);

/* host-buffer form of step(): fp32 actions from host memory, obs_f32/reward/done to host memory, synchronised before
 * returning. d_io is a caller-provided device buffer of sat_env_step_host_bytes(n) bytes. The inputs select the form:
 *   - all five host buffers pinned (UVA-mapped), rk4 mode and aux_stream != NULL: kernel A reads the actions from host
 *     memory and writes the next observation to d_io, from where a copy engine moves it to obs_host on aux_stream while
 *     kernel B runs on `stream` and writes reward / done straight to host memory;
 *   - all five pinned, any other case (cw mode, or aux_stream == NULL): zero-copy on `stream`, the kernels read the
 *     actions from and write the results to the host buffers directly;
 *   - otherwise (pageable memory): staged copies on `stream`: H2D of the actions to d_io, the step, D2H of the results. */
int64_t sat_env_step_host_bytes(int64_t n);
int sat_env_step_host(const SatEnvState* st, const float* pa_host, const float* ea_host,
                      float* obs_host, double* reward_host, uint8_t* done_host, void* d_io,
                      const SatEnvParams* p, void* stream, void* aux_stream);

/* ------------------------------------------------------------------------------------------------
 * Normalisation. Replaces RunningMeanStd.update / Normalization.__call__ (normalization.py:19-43)
 * for a batch x [n][dim] fp64: merge the batch into stats (Chan; n == 1 is the reference's Welford
 * step incl. its first-sample rule), then x_out = (x - mean) / (std + 1e-8). update = 0 only normalises.
 * ------------------------------------------------------------------------------------------------ */
int sat_norm_update(double* stats, const double* x, int64_t n, int dim, int update,
                    double* x_out_f64, float* x_out_f32, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Statistics shared across ranks. A batch sharded over G ranks keeps one set of running statistics: every rank computes
 * its per-block (mean, M2) partials, the partials of all ranks are gathered rank-major, and every rank folds all of them
 * into its own copy of the statistics. The fold is sat_env_step's / sat_norm_update's merge run over a block index that
 * spans the ranks in rank order, so every rank ends with the same bits.
 * Bit identity with the union batch: when every rank but the last holds a multiple of the rows per block (64 for the env
 * step, 128 for sat_norm_partials), rank r's blocks are exactly the union batch's blocks, and the statistics after the
 * fold are bit-identical to those one sat_env_step / sat_norm_update over the union batch leaves. Otherwise the blocks
 * straddle ranks differently and the result agrees with the union batch to rounding only (still the same on every rank).
 * ------------------------------------------------------------------------------------------------ */
/* bytes of one rank's partials for n rows: dim == 0, the env step's [ceil(n/64)][19][2] doubles (18 observation dims, then
 * the discounted return); 1 <= dim <= 32, sat_norm_partials' [ceil(n/128)][dim][2]. 0 for n <= 0 or another dim. */
int64_t sat_stats_partials_bytes(int64_t n, int dim);
/* sat_env_step with statistics on, except that the per-block partials are written to `partials`
 * (sat_stats_partials_bytes(n, 0) bytes) instead of being folded; no statistics are touched. workspace:
 * sat_workspace_bytes(n) bytes; the step zeroes its ticket (first 4 bytes), so it can be passed to sat_stats_fold next. */
int sat_env_step_partials(const SatEnvState* st, const void* pa, const void* ea, const int32_t* count_override,
                          float* obs_f32, double* obs_f64, double* term_obs_f64, double* reward, uint8_t* done,
                          double* partials, void* workspace, const SatEnvParams* p, void* stream);
/* the partials of a batch x [n][dim] fp64 (1 <= dim <= 32) into `partials` (sat_stats_partials_bytes(n, dim) bytes).
 * workspace: >= 256 bytes; its ticket (first 4 bytes) is zeroed. */
int sat_norm_partials(const double* x, int64_t n, int dim, double* partials, void* workspace, void* stream);
/* Fold the gathered partials of `ranks` ranks into the running statistics. partials: device, rank-major, rank r's block j
 * at ((r * rank_stride_blocks + j) * dims + d) * 2 (dims = 19 for dim == 0, else dim); rank_rows: device int64 [ranks],
 * rank r's row count, 0 <= rank_rows[r] <= rank_stride_blocks * rows per block.
 *   dim == 0: env-step partials into obs_stats (dim 18) / ret_stats (dim 1) / ret_std_out, each nullable, as sat_env_step.
 *   dim >= 1: sat_norm_partials partials into obs_stats (dim `dim`); ret_stats and ret_std_out must be NULL.
 * workspace: its first 4 bytes (the ticket) must be 0 on entry and are 0 again on exit; the workspace just given to
 * sat_env_step_partials / sat_norm_partials on the same stream satisfies this. With ranks == 1 the fold produces the bits
 * of sat_env_step's / sat_norm_update's own merge. Zero rows in total: the statistics are left unchanged. */
int sat_stats_fold(const double* partials, int ranks, int64_t rank_stride_blocks, const int64_t* rank_rows, int dim,
                   double* obs_stats, double* ret_stats, double* ret_std_out, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K3  fused Gaussian actor. Replaces PPO_continuous.choose_action -> Actor_Gaussian.get_dist/forward
 * (ppo_continuous.py:83-95, 176-189) over n observations: mean = max_action*tanh(W3 tanh(W2 tanh(W1 s+b1)+b2)+b3),
 * a = clamp(mean + exp(log_std)*eps, +-max_action), logp = Normal(mean, std).log_prob(a) per dimension.
 * eps comes from Philox4x32-10 keyed by (seed, global row id, step) unless eps_in is given.
 * Only the reference's network shape is supported: in_dim 18, hidden 256, act_dim 3 (SAT_ERR_SIZE otherwise).
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
    const float* w1;      /* fc1.weight        [hidden][in_dim]  (torch layout) */
    const float* b1;      /* fc1.bias          [hidden] */
    const float* w2;      /* fc2.weight        [hidden][hidden] */
    const float* b2;      /* fc2.bias          [hidden] */
    const float* w3;      /* mean_layer.weight [act_dim][hidden] */
    const float* b3;      /* mean_layer.bias   [act_dim] */
    const float* log_std; /* [act_dim] (NULL for the critic) */
    const float* packed;  /* device buffer of SAT_ACTOR_PACKED_FLOATS floats filled by sat_actor_pack() */
    int32_t in_dim, hidden, act_dim;   /* 18, 256, 3 (critic: act_dim = 1) */
    int32_t use_tanh;                  /* activation: 1 tanh (args.use_tanh, ppo_continuous.py:74), 0 ReLU */
    float   max_action;                /* 1.6 */
} SatActorWeights;

/* kernel-side weight image: W1^T [18][256], b1, W2^T [256][256] (k-major, streamed by TMA bulk copies),
 * b2, heads [4][256], b3[4], log_std[4]. Re-pack after every optimiser step (one tiny launch). */
#define SAT_ACTOR_PACKED_FLOATS (18 * 256 + 256 + 256 * 256 + 256 + 4 * 256 + 4 + 4)
int sat_actor_pack(const SatActorWeights* w, float* packed, void* stream);

/* obs source: either obs_f32 [n][18], or (obs_f32 == NULL) the env state itself, in which case the
 * observation is rebuilt from the fp64 SoA state and, when obs_stats != NULL, normalised in fp64 with
 * (x - mean)/(std + 1e-8) before the cast to fp32 (the fused path). obs_out (nullable) receives the
 * fp32 observation actually fed to the network. row_offset is the global id of row 0 (sharding). */
int sat_actor_sample(const SatActorWeights* w, const float* obs_f32, const SatEnvState* st,
                     const double* obs_stats, int64_t n, int64_t row_offset, uint64_t seed, uint64_t step,
                     const float* eps_in, float* act, float* logp, float* mean_out, float* eps_out,
                     float* obs_out, void* stream);

/* Critic forward (ppo_continuous.py:123-128): v [n] = fc3(tanh(fc2(tanh(fc1(s))))).
 * w3/b3 are fc3.weight [1][hidden] / fc3.bias [1]; log_std unused. */
/* The same sampling call with both dense layers on the tensor cores (csrc/actor_tc.cu): every fp32 operand is split exactly
 * into three bf16 words and six tcgen05.mma products are accumulated in fp32 in TMEM (the exact 16-bit A_h B_h products in their
 * own accumulator), so the result carries fp32-level accuracy like the reference's fp32 forward (ppo_continuous.py:83-95);
 * tests/test_gpu_actor_tc.py holds its error against an fp64 ground truth at or below the FFMA path's. Same arguments and
 * Philox stream as sat_actor_sample; tc_image is a caller-owned device scratch of SAT_ACTOR_TC_IMAGE_FLOATS floats (the
 * pre-split, pre-swizzled weight operands; rebuilt from w->packed on every call, so it is never stale). sm_100a only.
 * sat_actor_sample_pair_tc: two networks (same activation) on the same observations in ONE persistent launch, exactly the
 * results of two sat_actor_sample_tc calls with steps step_a / step_b (the tensor-core form of sat_actor_sample_pair). */
#define SAT_ACTOR_TC_IMAGE_FLOATS (2 * 256 * 256)
int sat_actor_sample_tc(const SatActorWeights* w, float* tc_image, const float* obs_f32, const SatEnvState* st,
                        const double* obs_stats, int64_t n, int64_t row_offset, uint64_t seed, uint64_t step,
                        const float* eps_in, float* act, float* logp, float* mean_out, float* eps_out, float* obs_out,
                        void* stream);
int sat_actor_sample_pair_tc(const SatActorWeights* wa, const SatActorWeights* wb, float* tc_image_a, float* tc_image_b,
                             const float* obs_f32, const SatEnvState* st, const double* obs_stats, int64_t n, int64_t row_offset,
                             uint64_t seed, uint64_t step_a, uint64_t step_b, float* act_a, float* logp_a, float* obs_out,
                             float* act_b, float* logp_b, void* stream);
/* Opponent pool (self-play against past snapshots): the learner wa on all n rows and, on contiguous groups of rows, frozen
 * snapshots of earlier networks, all in ONE persistent launch (the learner's tiles, then every group's tiles).
 * sat_actor_tc_snapshot builds a snapshot of w once: its tensor-core weight image (tc_image, SAT_ACTOR_TC_IMAGE_FLOATS
 * floats) and its bias / head tables (tc_tables, SAT_ACTOR_TC_TABLE_FLOATS floats), both from w->packed, and fills *snap
 * (host memory) with the pointers, w's activation and max_action; row_end is left 0. w->packed, tc_image and tc_tables must
 * stay unchanged while the snapshot is in use (copy the packed weights first if the network trains on).
 * sat_actor_sample_pool_tc: group k covers rows [groups_host[k - 1].row_end, groups_host[k].row_end) (0 for k = 0); its
 * outputs act_b / logp_b are exactly those of sat_actor_sample_tc of that snapshot on those rows with row offset
 * row_offset + groups_host[k - 1].row_end and step step_b; act_a / logp_a / obs_out are exactly sat_actor_sample_pair_tc's
 * net-a outputs. 1 <= groups <= SAT_ACTOR_POOL_MAX_GROUPS, row_end strictly increasing, every row_end but the last a multiple
 * of 128 (the row tile) and the last = n (SAT_ERR_SIZE); every snapshot built with wa's activation (SAT_ERR_MODE). */
#define SAT_ACTOR_POOL_MAX_GROUPS 16
#define SAT_ACTOR_TC_TABLE_FLOATS (5 * 256)   /* per column pair two float4 (b2, head weights), then b1 in accumulator order */
typedef struct {
    const float* packed;      /* the snapshot's SAT_ACTOR_PACKED_FLOATS weights (b3 and log_std are read from here) */
    const float* tc_image;    /* its tensor-core weight image */
    const float* tc_tables;   /* its bias / head tables */
    int64_t row_end;          /* exclusive end of the group's rows (set by the caller before sampling) */
    int32_t use_tanh;         /* activation the snapshot was built with */
    float   max_action;
} SatActorPoolGroup;
int sat_actor_tc_snapshot(const SatActorWeights* w, float* tc_image, float* tc_tables, SatActorPoolGroup* snap, void* stream);
int sat_actor_sample_pool_tc(const SatActorWeights* wa, float* tc_image_a, const SatActorPoolGroup* groups_host, int groups,
                             const float* obs_f32, const SatEnvState* st, const double* obs_stats, int64_t n,
                             int64_t row_offset, uint64_t seed, uint64_t step_a, uint64_t step_b, float* act_a, float* logp_a,
                             float* obs_out, float* act_b, float* logp_b, void* stream);
int sat_critic_forward(const SatActorWeights* w, const float* obs_f32, int64_t n, float* v, void* stream);
/* Two Gaussian actors on the same observations in ONE launch (pursuer and evader of a rollout step, CPPO_main.py:122-123):
 * exactly the results of two sat_actor_sample calls with steps step_a / step_b; obs_out (nullable) receives the fp32
 * observation once. At small shard sizes both networks then share the GPU instead of running one after the other. */
int sat_actor_sample_pair(const SatActorWeights* wa, const SatActorWeights* wb, const float* obs_f32, const SatEnvState* st,
                          const double* obs_stats, int64_t n, int64_t row_offset, uint64_t seed, uint64_t step_a,
                          uint64_t step_b, float* act_a, float* logp_a, float* obs_out, float* act_b, float* logp_b,
                          void* stream);


/* ------------------------------------------------------------------------------------------------
 * K4  GAE reverse scan. Replaces the block at ppo_continuous.py:198-210.
 * time-major form: r, done [T][N]; v [T+1][N] with v[t+1] = V(s') of step t (dw == done, SURVEY Q8);
 * r_scale nullable [T]: per-step reward scale (1/(std_R+1e-8)) applied on the fly.
 * gamma, lamda are the reference's python floats: the recursion coefficient is their double product rounded to fp32
 * (gamma*lamda*gae under numpy 2), the delta uses gamma rounded to fp32 (torch's fp32 tensor times a python float).
 * flat form: the reference's (B,1) buffers of one env in time order, with separate vs_next and dw.
 * Outputs adv / v_target share the input layout. sat_adv_normalize applies
 * (adv - mean)/(std_unbiased + 1e-5) (ppo_continuous.py:210); sums[3] (nullable in/out) lets the caller
 * all-reduce (sum, sum of squares, count) across ranks between the two phases.
 * ------------------------------------------------------------------------------------------------ */
int sat_gae(const float* r, const float* v, const uint8_t* done, const float* r_scale, int64_t T, int64_t N,
            double gamma, double lamda, float* adv, float* v_target, void* stream);
int sat_gae_flat(const float* r, const float* vs, const float* vs_next, const float* dw, const float* done,
                 int64_t B, double gamma, double lamda, float* adv, float* v_target, void* stream);
int sat_adv_moments(const float* adv, int64_t count, double* sums /*[3] device*/, void* workspace, void* stream);
int sat_adv_normalize(float* adv, int64_t count, const double* sums /*[3] device*/, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Batched forms of the satellite_function.py / RK4-script helpers the drop-in facade exposes.
 * ------------------------------------------------------------------------------------------------ */
/* StateEq(t, RV) ("轨道外推-龙格库塔算法.py":15-30): f [6][ld] = [v, a(x)] for n states x [6][ld]. */
int sat_state_eq(const double* x, double* f, int64_t n, int64_t ld, double mu, double re, double j2, void* stream);
/* Clohessy_Wiltshire(...).State_transition_matrix(t) (satellite_function.py:753-781): x [6][ld] <- M x with
 * numpy's dgemv summation order; stm_host is the row-major 6x6 matrix in HOST memory (copied into the launch). */
int sat_cw_propagate(double* x, int64_t n, int64_t ld, const double* stm_host, void* stream);
/* Numerical_calculation_method(...).numerical_calculation(t) (satellite_function.py:783-839): the CW ODE (orbit_ode,
 * :793-821, thrust = J2 = 0) integrated from 0 to t_bound by scipy's adaptive RK45 (Dormand-Prince 5(4), scipy 1.18.1
 * step control restated), value at t_bound, for n states x [6][ld] in place. w2 = 2*omega, w3 = 3*omega**2,
 * wz = omega**2 as python computes them; rtol/atol = solve_ivp's 1e-3 / 1e-6. status_out (nullable) [n]: 0, or -1
 * where scipy would stop with "step size too small". */
int sat_cw_ode_rk45(double* x, int64_t n, int64_t ld, double t_bound, double w2, double w3, double wz,
                    double rtol, double atol, int32_t* status_out, void* stream);
/* calculate_orbital_elements(miu, R0, V0) (satellite_function.py:161-255): rv [n][6] -> (a,e,i,omega,Omega,f) [n][6];
 * kind_out [n] = 6, or 0 (elements_out unspecified) for the circular / parabolic element sets: sat_orbital_elements_all
 * returns those. */
int sat_orbital_elements(const double* rv, int64_t n, double miu, double* elements_out, int32_t* kind_out, void* stream);
/* calculate_state_information(data, miu) (satellite_function.py:257-315), six-element form: -> rv [n][6]. */
int sat_state_from_elements(const double* elements, int64_t n, double miu, double* rv_out, void* stream);
/* calculate_orbital_elements on every branch: elements_out [n][6] holds the list the reference returns, zero-padded, and
 * kind_out [n] its length, which names the branch (SAT_ELEM_KIND_*):
 *   SAT_ELEM_KIND_GENERAL   6: columns 0-5 = a, e, i, omega, Omega, f   (energy != 0 and e != 0: elliptic / hyperbolic;
 *                              the same bits as sat_orbital_elements)
 *   SAT_ELEM_KIND_PARABOLIC 5: columns 0-4 = p, i, omega, Omega, f      (energy == 0 exactly; column 5 = 0)
 *   SAT_ELEM_KIND_CIRCULAR  4: columns 0-3 = a, i, u, Omega             (e == 0 exactly; u = argument of latitude, NaN for
 *                              an equatorial orbit as in the reference; columns 4-5 = 0)
 * Bit-identical to the reference's arithmetic on every branch (the host libm's acos and pow, csrc/glibm.cuh). */
#define SAT_ELEM_KIND_GENERAL 6
#define SAT_ELEM_KIND_PARABOLIC 5
#define SAT_ELEM_KIND_CIRCULAR 4
int sat_orbital_elements_all(const double* rv, int64_t n, double miu, double* elements_out, int32_t* kind_out,
                             void* stream);
/* calculate_state_information(data, miu) for n element sets of n_el elements each, elements [n][n_el] -> rv [n][6]:
 *   n_el = 6: (a, e, i, omega, Omega, f), exactly sat_state_from_elements;
 *   n_el = 5: (p, i, omega, Omega, f), the parabolic form (e = 1);
 *   n_el = 4: (a, i, u, Omega), the circular form (e = 0).
 * The 5- and 4-element forms use the host libm's sin, cos and pow (csrc/glibm.cuh). Any other n_el: SAT_ERR_SIZE. */
int sat_state_from_elements_n(const double* elements, int64_t n, int n_el, double miu, double* rv_out, void* stream);

/* Reachable-domain sweep (SURVEY.md s8 f.3). Replaces Reachable_Domain() of single_pluse_model/RD_single_pulse.py:40-148
 * (N1 = 1) for n pursuer states given as elements [n][6] = (a, e, i, omega, Omega, f) and delta_max [n]: for each of the
 * (N2+1)*(N3+1) directions (i major, j minor - the reference's loop order) the reachability test and the two fsolve
 * extremes. rf_max / rf_min [n][(N2+1)*(N3+1)][3] = max / min |rf| times the direction vector, valid [n][...] = 1 for the
 * directions the reference appends to its point clouds. The ellipse fit that follows upstream is out of scope. n <= 65535. */
int sat_reachable_domain(const double* elements, const double* delta_max, int64_t n, int N2, int N3, double u,
                         double* rf_max, double* rf_min, uint8_t* valid, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused PPO minibatch step (SURVEY.md s8 f.1). Replaces the body of the K-epoch loop of PPO_continuous.update
 * (ppo_continuous.py:216-239): actor clipped-surrogate + entropy loss, critic MSE loss, their backward passes through
 * the 18-256-256-{3,1} MLPs, clip_grad_norm_ and the Adam step (:161-163). fp32 CUDA-core FFMA2, no tensor cores.
 *
 * One network's parameters live in ONE flat fp32 buffer in torch parameter order (fc1.weight [256][18], fc1.bias,
 * fc2.weight [256][256], fc2.bias, mean_layer/fc3.weight [heads][256], bias [heads], log_std [3] for the actor), so the
 * torch modules can hold views of it and the gradient all-reduce is one NCCL call on `grads`. */
enum { SAT_PPO_OFF_W1 = 0, SAT_PPO_OFF_B1 = 4608, SAT_PPO_OFF_W2 = 4864, SAT_PPO_OFF_B2 = 70400, SAT_PPO_OFF_W3 = 70656 };
#define SAT_PPO_PARAM_FLOATS(heads) (70656 + 257 * (heads) + ((heads) == 3 ? 3 : 0))   /* actor 71430, critic 70913 */

typedef struct SatPpoNet {
    float* params;      /* flat parameters (SAT_PPO_OFF_*), updated in place by sat_ppo_adam; 16-byte aligned */
    float* packed;      /* SAT_ACTOR_PACKED_FLOATS kernel image of params (what sat_actor_sample reads); rewritten by sat_ppo_adam */
    float* grads;       /* flat gradient, same layout, SAT_PPO_PARAM_FLOATS + 1 floats: the last one is the minibatch loss
                           (SAT_PPO_GRAD_FLOATS_STATS for sat_ppo_actor_grad_stats) */
    float* exp_avg;     /* Adam first moment, flat */
    float* exp_avg_sq;  /* Adam second moment, flat */
    float* workspace;   /* sat_ppo_workspace_floats(mb) floats, may be shared by the two networks of one agent */
    int32_t heads;      /* 3 = Actor_Gaussian, 1 = Critic */
    int32_t use_tanh;   /* hidden activation: 1 tanh, 0 ReLU */
    float max_action;
    int32_t reserved;
} SatPpoNet;

/* Forward / backward kernel of sat_ppo_actor_grad / sat_ppo_critic_grad: tensor cores (csrc/ppo_fb_tc.cu: the three 256-wide
 * contractions per row tile as exact bf16x3 splits on tcgen05, fp32-level accuracy; the default) or the fp32 FFMA2 kernel
 * (enable = 0, or SAT_PPO_TC=0 in the environment). enable < 0 only queries. Returns the previous setting. Process-wide. */
int sat_ppo_use_tensor_cores(int enable);
int64_t sat_ppo_workspace_floats(int64_t mb);
/* rebuild `packed` from `params` (after loading a checkpoint into the torch views) */
int sat_ppo_pack(const SatPpoNet* net, void* stream);
/* gradient of mean(-min(ratio*adv, clamp(ratio, 1-eps, 1+eps)*adv) - entropy_coef*entropy) over the minibatch rows
 * index[0..mb) of s [B][18], a [B][3], old_logp [B][3], adv [B] (index == NULL: rows 0..mb) -> net->grads */
int sat_ppo_actor_grad(const SatPpoNet* net, const float* s, const float* a, const float* old_logp, const float* adv,
                       const int64_t* index, int64_t mb, float epsilon, float entropy_coef, void* stream);
/* gradient of mse_loss(v_target[index], critic(s[index])) -> net->grads */
int sat_ppo_critic_grad(const SatPpoNet* net, const float* s, const float* v_target, const int64_t* index, int64_t mb,
                        void* stream);
/* grads *= grad_scale (1/world after an all-reduce); clip_grad_norm_(max_grad_norm) when max_grad_norm > 0; Adam with
 * the learning rate read from device memory (*lr) and the step counter *step (device, incremented here) */
int sat_ppo_adam(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm,
                 float grad_scale, int64_t* step, void* stream);
/* The same step with the gradient all-reduce fused in (multi-GPU, SURVEY.md s8e exchange step 1): peer_grads is a DEVICE
 * array of `world` pointers to every rank's flat gradient buffer mapped into this process (NVLink peer memory, e.g. a
 * torch symmetric-memory allocation); the kernel reads peer_grads[r][offset_floats + i] for all r in rank order, so all
 * replicas compute bit-identical sums. The caller orders the ranks with a device-side barrier between the gradient
 * kernels and this call and alternates offset_floats between two halves of the buffer from step to step. */
int sat_ppo_adam_peers(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm,
                       float grad_scale, int64_t* step, const float* const* peer_grads, int world, int64_t offset_floats,
                       void* stream);

/* Training diagnostics of the fused step. sat_ppo_actor_grad_stats computes exactly the gradient and loss of
 * sat_ppo_actor_grad (bit-identical grads[0 .. n]) and also writes the minibatch means of four per-row terms to the tail
 * grads[n + 2 .. n + 6), n = SAT_PPO_PARAM_FLOATS(3): -min(surr1, surr2), the entropy, the approximate KL
 * (ratio - 1) - log ratio, and the fraction of rows with |ratio - 1| > epsilon. net->grads must then hold
 * SAT_PPO_GRAD_FLOATS_STATS(3) floats. Because the tail sits in the gradient buffer, an all-reduce of those floats (or the
 * peer read of sat_ppo_adam_peers_stats) carries the diagnostics with the gradient, and every rank sees the same sums.
 * sat_ppo_adam_stats / sat_ppo_adam_peers_stats do exactly the step of sat_ppo_adam / sat_ppo_adam_peers (bit-identical
 * parameters and moments) and, before it, ADD one minibatch to the device fp64 record [SAT_PPO_STATS_DOUBLES]: the loss
 * slot grads[n] and (actor only: heads == 3) the four tail terms, each times grad_scale (the global minibatch means after an
 * all-reduce), the pre-clip gradient norm, the clip coefficient and a count of 1. The caller zeroes the record; per-epoch
 * means are sum / count. */
#define SAT_PPO_GRAD_FLOATS_STATS(heads) (SAT_PPO_PARAM_FLOATS(heads) + 6)
#define SAT_PPO_STAT_LOSS 0        /* minibatch loss: actor surrogate - entropy_coef * entropy, or the critic's MSE */
#define SAT_PPO_STAT_SURROGATE 1   /* actor: mean of -min(ratio * adv, clamp(ratio, 1 - eps, 1 + eps) * adv) */
#define SAT_PPO_STAT_ENTROPY 2     /* actor: mean entropy of the Gaussian policy (summed over the action dimensions) */
#define SAT_PPO_STAT_APPROX_KL 3   /* actor: mean of (ratio - 1) - log ratio, evaluated as expm1(log ratio) - log ratio */
#define SAT_PPO_STAT_CLIP_FRAC 4   /* actor: fraction of rows with |ratio - 1| > epsilon */
#define SAT_PPO_STAT_GRAD_NORM 5   /* global gradient norm before clipping (what clip_grad_norm_ returns) */
#define SAT_PPO_STAT_CLIP_COEF 6   /* gradient scale applied by the clip: min(max_norm / (norm + 1e-6), 1), 1 without clip */
#define SAT_PPO_STAT_COUNT 7       /* number of minibatches added */
#define SAT_PPO_STATS_DOUBLES 8
int sat_ppo_actor_grad_stats(const SatPpoNet* net, const float* s, const float* a, const float* old_logp, const float* adv,
                             const int64_t* index, int64_t mb, float epsilon, float entropy_coef, void* stream);
int sat_ppo_adam_stats(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm,
                       float grad_scale, int64_t* step, double* record, void* stream);
int sat_ppo_adam_peers_stats(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm,
                             float grad_scale, int64_t* step, const float* const* peer_grads, int world, int64_t offset_floats,
                             double* record, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Measurement helpers (bench.py): dependent-free DFMA / FFMA chains to measure the FP64 / FP32
 * vector peaks on the device the bench runs on (MEASURED_PEAKS.json has no such entries).
 * Each launches one kernel doing `iters` x 16 independent FMAs per thread; flops_out (host) receives
 * the FLOP count of the launch.
 * ------------------------------------------------------------------------------------------------ */
int sat_peak_fp64(double* sink, int blocks, int threads, int iters, double* flops_out_host, void* stream);
int sat_peak_fp32(float* sink, int blocks, int threads, int iters, double* flops_out_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SATB200_H */
