/*
 * sat_oracle.h -- CPU restatement of the PPO-RL-Satellite hot path (TEST INFRASTRUCTURE ONLY).
 *
 * This library is the parity checker for the CUDA path. It is NOT shipped and is never
 * imported by the product package: only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load it.
 *
 * Every function cites the reference file:line (paths relative to the upstream repository
 * qiaobeibei/PPO-RL-Satellite) whose arithmetic it restates. The restatement is pinned by
 * tests/test_oracle_golden.py against fixtures produced by running the reference itself
 * (tests/golden/make_golden.py) and against the reference's own known-answer data
 * (single_pluse_model/spacecraft_state.txt <-> all_input.csv, and the RK4 script's initial
 * condition).
 *
 * Third-party arithmetic restated from its published algorithm:
 *   - scipy.optimize.fsolve -> MINPACK hybrd (n = 1), scipy 1.18.1 defaults
 *   - numpy/OpenBLAS 0.3.30 (Haswell kernels) summation order of ddot / dgemv for the 3- and
 *     6-element products the env performs (needed for bit-identical states and rewards).
 */
#ifndef SAT_ORACLE_H
#define SAT_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- RK4 two-body + J2 (reference script "轨道外推-龙格库塔算法.py":15-40) ---- */
void orc_state_eq(const double rv[6], double mu, double re, double j2, double f[6]);
void orc_rk4_step(double rv[6], double h, double mu, double re, double j2);
/* x is SoA [6][ld]; propagates n states by `steps` RK4 steps of size h using nthreads OpenMP threads */
void orc_rk4_batch(double* x, int64_t n, int64_t ld, double h, int steps,
                   double mu, double re, double j2, int nthreads);

/* ---- Clohessy-Wiltshire STM (satellite_function.py:744-781) ---- */
void orc_cw_matrix(double t, double M[36]);
void orc_cw_apply(const double M[36], const double s[6], double out[6]); /* np.dot(matrix, state) order */

/* ---- small BLAS-order helpers (numpy/OpenBLAS emulation) ---- */
double orc_dot3(const double a[3], const double b[3]);
double orc_norm3(const double a[3]);

/* ---- orbital elements / state (satellite_function.py:161-255, 257-315) ---- */
/* returns number of elements written (6 elliptic/hyperbolic, 5 parabolic, 4 circular) */
int  orc_orbital_elements(double miu, const double R0[3], const double V0[3], double out[6]);
void orc_state_information(const double el[6], double miu, double R[3], double V[3]);

/* ---- fsolve for n = 1 (MINPACK hybrd, SURVEY.md Appendix B) ---- */
typedef double (*orc_fn1)(double x, void* ctx);
double orc_fsolve1(orc_fn1 f, void* ctx, double x0, int* nfev_out, int* info_out);
/* P_fai_equation root (satellite_function.py:558-565) */
double orc_numerical_iteration(double u, double Delta_Vm, double theta, double v_1x, double v_1y,
                               double h, double alpha_guess);

/* ---- danger-zone count (satellite_function.py:18-99, 317-373, 462-565) ---- */
/* returns 0/1/2, or -1 when the reference would raise (circular / parabolic element sets) */
int orc_danger_zone(const double R0_c[3], const double V0_c[3], const double R0_t[3], const double V0_t[3],
                    double Delta_V_c, double u);
int orc_danger_zone_debug(const double R0_c[3], const double V0_c[3], const double R0_t[3], const double V0_t[3],
                          double Delta_V_c, double u, double* dbg /* nullable [2][8] */);

/* ---- environment (environment.py:26-179 Flag 0, :181-255 Flag 1, :317-396) ---- */
typedef struct {
    double P[3], Pv[3], E[3], Ev[3];
    double fuel_c, fuel_t, dis;
    int32_t dangerous_zone;
    int32_t int_state;      /* 1 right after reset(): arrays are int64 (Q1 truncation on next step) */
    int32_t flag;           /* 0 pursuer training, 1 evader training */
    int32_t err;            /* sticky: 1 if the reference would have raised in the danger-zone code */
    double d_capture, d_range;
    int32_t max_episode_steps;
} orc_env;

void orc_env_init(orc_env* e, double d_capture, double d_range, double fuel_c, double fuel_t,
                  int max_episode_steps);
void orc_env_reset(orc_env* e, int flag, double obs[18]);
/* M = STM for the 100 s step (pass orc_cw_matrix(100) or the numpy-computed one). returns done */
int  orc_env_step(orc_env* e, const double M[36], const double pa[3], const double ea[3],
                  int episode_count, double obs[18], double* reward);
/* per-term breakdown of the last non-terminal reward, for diagnostics: a,b,c,pv1..pv4 */
void orc_env_last_terms(double out[7]);

/* batched driver used as the CPU baseline: n independent envs (AoS array), one step each with
 * auto-reset, actions [n][3]; uses nthreads OpenMP threads. */
void orc_env_step_batch(orc_env* envs, int32_t* counts, int64_t n, const double M[36],
                        const double* pa, const double* ea, double* obs /*[n][18]*/,
                        double* reward, uint8_t* done, int auto_reset, int nthreads);

/* env step whose propagation is S RK4 substeps in the inertial frame (SURVEY H8; no upstream env) */
int  orc_env_step_rk4(orc_env* e, double h, int substeps, double mu, double re, double j2,
                      const double pa[3], const double ea[3], int episode_count,
                      double obs[18], double* reward);
void orc_env_step_rk4_batch(orc_env* envs, int32_t* counts, int64_t n, double h, int substeps,
                            double mu, double re, double j2, const double* pa, const double* ea,
                            double* obs, double* reward, uint8_t* done, int auto_reset, int nthreads);

/* ---- Numerical_calculation_method.numerical_calculation (satellite_function.py:793-839): scipy RK45 on the CW ODE;
 * y in/out, returns 0 or -1 (step too small) ---- */
int orc_cw_ode_rk45(double y[6], double t_bound, double w2, double w3, double wz, int* nsteps_out);

/* ---- reachable-domain sweep (single_pluse_model/RD_single_pulse.py:40-148, N1 = 1); outputs [(N2+1)*(N3+1)][3] and a mask ---- */
void orc_reachable_domain(const double el[6], double delta_max, int N2, int N3, double u,
                          double* rf_max_xyz, double* rf_min_xyz, uint8_t* valid);

/* ---- normalisation (normalization.py:7-63) ---- */
typedef struct { int64_t n; int dim; double* mean; double* S; double* std; } orc_rms;
void orc_rms_update(orc_rms* r, const double* x);                       /* :19-29 incl. n==1 rule */
void orc_normalize(orc_rms* r, const double* x, int update, double* out); /* :37-43 */
double orc_reward_scaling(orc_rms* r, double* R, double gamma, double x);  /* :56-60 (shape 1) */

/* ---- GAE (ppo_continuous.py:198-210); fp32 recursion as executed under numpy 2 ---- */
void orc_gae(const float* r, const float* vs, const float* vs_next, const float* dw, const float* done,
             int64_t B, double gamma, double lamda, float* adv, float* v_target);
void orc_adv_normalize(float* adv, int64_t B); /* (adv-mean)/(std_unbiased+1e-5), torch semantics */

/* ---- Gaussian actor (ppo_continuous.py:83-95, 176-189), fp32 ---- */
void orc_actor_forward(const float* W1, const float* b1, const float* W2, const float* b2,
                       const float* W3, const float* b3, int in_dim, int hid, int act_dim,
                       float max_action, const float* s, int64_t n, float* mean);
void orc_gaussian_sample(const float* mean, const float* log_std, const float* eps, int64_t n, int act_dim,
                         float max_action, float* a, float* logp);
void orc_critic_forward(const float* W1, const float* b1, const float* W2, const float* b2,
                        const float* W3, const float* b3, int in_dim, int hid,
                        const float* s, int64_t n, float* v);

#ifdef __cplusplus
}
#endif
#endif
