// env_step.cu -- K2: fused batched satellites.step()/reset() for sm_100a.
//
// Reference behaviour replaced (paths relative to the upstream repo):
//   environment.py:66-79 (reset), :81-179 (step, Flag 0), :181-255 (step, Flag 1),
//   :317-343 (danger-zone count, relative->inertial), :346-396 (reward cosines),
//   satellite_function.py:744-781 (CW STM), :18-99,161-255,317-373,462-565 (danger zone + fsolve),
//   normalization.py:19-29,56-60 (running statistics of observations / discounted returns).
//
// Mapping: TWO lanes per environment (even lane = pursuer, odd lane = escaper). Each lane owns one
// craft through impulse + propagation + orbital elements, the pair exchanges results with
// __shfl_xor(…, 1), and each lane then sets up one of the two relative-node reachability problems;
// the fsolve work items are compacted across the CTA through a shared-memory queue.
//   cw  mode: ONE kernel (propagation is a 6x6 product).
//   rk4 mode: kernel A = clip/gate/impulse + S RK4 substeps in registers (FP64-pipe bound, 72 registers,
//             64-thread CTAs so the whole 65 536-env batch (2048 CTAs) is resident at 14 CTAs/SM);
//             kernel B = everything after the propagation (register-heavy, divergent). The split costs one
//             extra read of the state (~130 B/env, ~1 us at 65 536 envs) and lets each half run at its own
//             occupancy.
//
// Data layout in HBM: SoA fp64 columns [16][ld] + int32 columns [4][ld] (include/satb200.h).
// Compiled with -fmad=false: the env arithmetic must round exactly like numpy's.
#include "sat_math.cuh"
#include "../../include/satb200.h"
#include <cmath>

namespace {

using namespace sat;

constexpr int kBlock = 128;             // finish / fused kernels: threads per CTA (2 lanes per env)
constexpr int kEnvsPerBlock = kBlock / 2;
constexpr int kFrontBlock = 64;         // rk4 front (impulse + propagation) kernel
// kernel B is latency bound (long dependent FP64 chains: divisions, sqrt, acos, sincos): measured on B200 at 65 536
// envs, total env-step time vs min-blocks-per-SM {1: 250, 4: 200, 7: 185, 8: 187, 10: 201, 12: 231} us. 7 CTAs x 128
// threads at 72 registers (some spills to L1) beats 186 registers at 2 CTAs.
#ifndef SAT_FINISH_MINB
#define SAT_FINISH_MINB 7
#endif
constexpr int kFinishMinBlocks = SAT_FINISH_MINB;
constexpr int kObs = 18;
constexpr int kStatDims = 19;           // 18 observation dims + discounted return
constexpr int kWsHeader = 256;          // workspace: [ticket counter | pad] [dis_prev: n doubles] [partials]

SAT_DEV double shfl1(double v) { return __shfl_xor_sync(0xffffffffu, v, 1); }
SAT_DEV int shfl1(int v) { return __shfl_xor_sync(0xffffffffu, v, 1); }

SAT_DEV double clip16(double a) { return a < -1.6 ? -1.6 : (a > 1.6 ? 1.6 : a); }   // np.clip, environment.py:86-87

__host__ __device__ inline int64_t ws_disprev_offset() { return kWsHeader; }
__host__ __device__ inline int64_t ws_partials_offset(int64_t n) { return kWsHeader + ((n * 8 + 255) / 256) * 256; }

// ---------------------------------------------------------------------------------------------
// front half of step(): clip, gate, impulse (with the int64 truncation quirk), fuel, propagation of the
// lane's own craft. environment.py:86-121 (Flag 0) / :185-210 (Flag 1).
// ---------------------------------------------------------------------------------------------
struct Lane {
    double r[3], v[3];      // own craft, relative frame
    double a[3];            // own clipped + gated action
    double fuel_own;
    double dis_prev;        // |P - E| before the step (:89)
};

template <typename ActT>
SAT_DEV void load_and_gate(const SatEnvState& st, const SatEnvParams& p, const ActT* __restrict__ pa,
                           const ActT* __restrict__ ea, int64_t e, int craft, Lane& L, bool do_impulse,
                           const ActT* raw = nullptr /* the lane's action already in registers */) {
    const int64_t ld = st.ld;
    const double* __restrict__ S = st.state;
    const int32_t* __restrict__ I = st.istate;
    const int base = craft * 6;
#pragma unroll
    for (int k = 0; k < 3; ++k) { L.r[k] = S[(base + k) * ld + e]; L.v[k] = S[(base + 3 + k) * ld + e]; }
    L.fuel_own = S[(SAT_COL_FUEL_C + craft) * ld + e];
    const double dis_stale = S[SAT_COL_DIS * ld + e];
    const int dz_stale = I[SAT_ICOL_DZ * ld + e];
    const int int_state = I[SAT_ICOL_INTSTATE * ld + e];
    {
        const ActT* act = craft ? ea : pa;
#pragma unroll
        for (int k = 0; k < 3; ++k) L.a[k] = clip16((double)(raw ? raw[k] : act[e * 3 + k]));
    }
    bool frozen;                                            // gating uses LAST step's dis / dangerous_zone (Q3)
    if (p.flag != 1) frozen = (craft == 0) && (dis_stale < p.d_range) && (dz_stale != 0);   // :91-96 (Flag 2: :265-277)
    else frozen = (craft == 1) && (dz_stale == 0);                                          // :190-198
    if (frozen) { L.a[0] = 0.0; L.a[1] = 0.0; L.a[2] = 0.0; }
    if (!do_impulse) return;
    double d[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double o = shfl1(L.r[k]);
        d[k] = craft == 0 ? __dsub_rn(L.r[k], o) : __dsub_rn(o, L.r[k]);
    }
    L.dis_prev = norm3(d);                                  // :89
    // right after reset() the arrays are int64 and `+=` truncates toward zero (Q1)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double s = __dadd_rn(L.v[k], L.a[k]);
        L.v[k] = int_state ? trunc(s) : s;
    }
    L.fuel_own = __dsub_rn(L.fuel_own, __dadd_rn(__dadd_rn(fabs(L.a[0]), fabs(L.a[1])), fabs(L.a[2])));   // :106-107
}

SAT_DEV void propagate_cw(const SatEnvParams& p, Lane& L) {
    const double x6[6] = {L.r[0], L.r[1], L.r[2], L.v[0], L.v[1], L.v[2]};
    double y6[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) y6[i] = gemv6_row(p.stm + 6 * i, x6);      // satellite_function.py:778-779
#pragma unroll
    for (int k = 0; k < 3; ++k) { L.r[k] = y6[k]; L.v[k] = y6[3 + k]; }
}

SAT_DEV void propagate_rk4(const SatEnvParams& p, Lane& L) {
    double X[3], V[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { X[k] = p.r_cw[k] + L.r[k]; V[k] = p.v_cw[k] + L.v[k]; }
    const Rk4Consts c = make_rk4_consts(p.h, p.mu, p.re, p.j2);
    if (p.j2 != 0.0) {
#pragma unroll 1
        for (int s = 0; s < p.substeps; ++s) rk4_step<true>(X, V, c);
    } else {
#pragma unroll 1
        for (int s = 0; s < p.substeps; ++s) rk4_step<false>(X, V, c);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { L.r[k] = X[k] - p.r_cw[k]; L.v[k] = V[k] - p.v_cw[k]; }
}

// rk4 mode, kernel A: impulse + S RK4 substeps, state written back; |P-E| before the step goes to the workspace.
// 64-thread CTAs at <= 72 registers: all 2048 CTAs of the 65 536-env batch are resident at once (14 per SM).
// OBS = true (host-buffer path): the kernel also writes the step's NEXT observation (after the auto reset) to obs_early.
// The observation depends only on the propagated state and the terminal checks, not on the danger-zone solve of kernel
// B, so its device-to-host copy can run on a copy engine underneath kernel B.
// STARTS (auto_reset == SAT_RESET_STARTS, OBS only): the post-reset observation comes from the env's start columns.
template <typename ActT, bool OBS, bool STARTS = false>
__global__ void __launch_bounds__(kFrontBlock, 14)
env_front_rk4_kernel(const SatEnvState st, const ActT* __restrict__ pa, const ActT* __restrict__ ea,
                     double* __restrict__ dis_prev_out, float* __restrict__ obs_early,
                     float* __restrict__ pa_copy, float* __restrict__ ea_copy, const __grid_constant__ SatEnvParams p) {
    const int64_t tid = (int64_t)blockIdx.x * kFrontBlock + threadIdx.x;
    const int64_t env_raw = tid >> 1;
    const int craft = (int)(tid & 1);
    const bool valid = env_raw < st.n;
    const int64_t e = valid ? env_raw : st.n - 1;
    Lane L;
    if (OBS) {
        // host-buffer path: pa / ea live in host memory. Each action is read over PCIe exactly once, here, and left in
        // device memory for kernel B - whose reads would otherwise queue behind the observation copy's posted writes
        // (PCIe ordering: a read request may not pass a write in the same direction)
        ActT raw[3];
        const ActT* act = craft ? ea : pa;
#pragma unroll
        for (int k = 0; k < 3; ++k) raw[k] = act[e * 3 + k];
        if (valid) {
            float* dc = craft ? ea_copy : pa_copy;
#pragma unroll
            for (int k = 0; k < 3; ++k) dc[e * 3 + k] = (float)raw[k];
        }
        load_and_gate(st, p, pa, ea, e, craft, L, true, raw);
    } else {
        load_and_gate(st, p, pa, ea, e, craft, L, true);
    }
    propagate_rk4(p, L);
    if (valid) {
        const int64_t ld = st.ld;
        const int base = craft * 6;
#pragma unroll
        for (int k = 0; k < 3; ++k) { st.state[(base + k) * ld + e] = L.r[k]; st.state[(base + 3 + k) * ld + e] = L.v[k]; }
        st.state[(SAT_COL_FUEL_C + craft) * ld + e] = L.fuel_own;
        if (craft == 0) dis_prev_out[e] = L.dis_prev;
    }
    if (OBS) {
        // same arithmetic as kernel B: exchange, |P - E|, terminal checks (environment.py:130-147), reset values (:66-79)
        double P[3], Pv[3], E[3], Ev[3], d[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double o_r = shfl1(L.r[k]), o_v = shfl1(L.v[k]);
            P[k] = craft == 0 ? L.r[k] : o_r;  Pv[k] = craft == 0 ? L.v[k] : o_v;
            E[k] = craft == 0 ? o_r : L.r[k];  Ev[k] = craft == 0 ? o_v : L.v[k];
            d[k] = __dsub_rn(P[k], E[k]);
        }
        const double dis = norm3(d);
        const int count_new = st.istate[SAT_ICOL_COUNT * st.ld + e] + 1;
        const bool done = (dis <= p.d_capture) || (count_new >= p.max_episode_steps);
        if (done && p.auto_reset) {
            if (STARTS) {
                // each lane loads the start columns itself: the lanes of one env agree on `done`, a warp does not
                const int64_t ld = st.ld;
                const double* __restrict__ Sst = st.state + SAT_COL_START * ld;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    P[k] = Sst[(SAT_COL_P + k) * ld + e]; Pv[k] = Sst[(SAT_COL_PV + k) * ld + e];
                    E[k] = Sst[(SAT_COL_E + k) * ld + e]; Ev[k] = Sst[(SAT_COL_EV + k) * ld + e];
                }
            } else {
#pragma unroll
                for (int k = 0; k < 3; ++k) { P[k] = p.reset_p[k]; E[k] = p.reset_e[k]; Pv[k] = 0.0; Ev[k] = 0.0; }
            }
        }
        if (valid) {
            float* o = obs_early + e * kObs + craft * 9;
            if (craft == 0) {
#pragma unroll
                for (int k = 0; k < 3; ++k) { o[k] = (float)__dsub_rn(P[k], E[k]); o[3 + k] = (float)__dsub_rn(Pv[k], Ev[k]); o[6 + k] = (float)P[k]; }
            } else {
#pragma unroll
                for (int k = 0; k < 3; ++k) { o[k] = (float)Pv[k]; o[3 + k] = (float)E[k]; o[6 + k] = (float)Ev[k]; }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// CTA-wide compaction of the fsolve work items: every lane with a reachable node pushes two root problems
// into a shared-memory queue; the queue is then processed densely (thread t <- task t), so warps beyond
// the task count skip the solver entirely instead of running it with ~1/4 of their lanes active.
// ---------------------------------------------------------------------------------------------
struct SolveQueue {
    double A[2 * kBlock], sth[2 * kBlock], dvm[2 * kBlock], alpha[2 * kBlock];
    int guess[2 * kBlock];
    double trig[2][4];      // per guess: sin, cos at x0 and at x0 + sqrt(eps)|x0| (Hybrd1::init_warm)
    int count, next;
};

template <bool EXACT = true>
SAT_DEV void queue_init(SolveQueue& q) {
    if (threadIdx.x == 0) { q.count = 0; q.next = 0; }
    if (threadIdx.x < 4) {
        const int j = threadIdx.x >> 1, k = threadIdx.x & 1;
        const double x0 = dz_guess(j);
        const double h = 1.4901161193847656e-08 * fabs(x0);           // Hybrd1::start_outer
        const double2 sc = Lm<EXACT>::sincos(k ? x0 + h : x0);
        q.trig[j][2 * k] = sc.x; q.trig[j][2 * k + 1] = sc.y;
    }
    __syncthreads();
}

// pushes the lane's non-degenerate root problems; returns their slots (-1: none / solved in place)
SAT_DEV void queue_push(SolveQueue& q, const DzNode& nd, int& slot0, int& slot1, double& alpha0, double& alpha1) {
    slot0 = -1; slot1 = -1; alpha0 = dz_guess(0); alpha1 = dz_guess(1);
    if (nd.status == 2) {
        const bool g0 = dz_degenerate(nd.A0, nd.sth, nd.dvm), g1 = dz_degenerate(nd.A1, nd.sth, nd.dvm);
        const int cnt = (g0 ? 0 : 1) + (g1 ? 0 : 1);
        if (cnt) {
            int s = atomicAdd(&q.count, cnt);
            if (!g0) { slot0 = s; q.A[s] = nd.A0; q.sth[s] = nd.sth; q.dvm[s] = nd.dvm; q.guess[s] = 0; ++s; }
            if (!g1) { slot1 = s; q.A[s] = nd.A1; q.sth[s] = nd.sth; q.dvm[s] = nd.dvm; q.guess[s] = 1; }
        }
    }
    __syncthreads();
}

// persistent lanes: every lane pulls the next root problem as soon as it finishes one, and all lanes of a warp
// advance their own solver by one function evaluation per loop trip (uniform loop body, no per-task divergence)
#ifndef SAT_SOLVE_WARPS
#define SAT_SOLVE_WARPS 4
#endif
template <bool EXACT = true>
SAT_DEV void queue_run(SolveQueue& q) {
    const int total = q.count;
    int task = -1;
    Hybrd1<PFaiT<EXACT>> hs;
    // root problems take 5..15 evaluations (mean 8), so a warp runs as long as its slowest lane (12.8 trips measured).
    // Restricting the solve to fewer warps evens the lanes out but lengthens the CTA's serial chain; the kernel is
    // latency-bound, so all four warps is fastest (env step 174 / 176 / 181 / 209 us with 4 / 3 / 2 / 1 solver warps).
    if ((threadIdx.x >> 5) < SAT_SOLVE_WARPS)
    for (;;) {
        if (task < 0) {
            const int t = atomicAdd(&q.next, 1);
            if (t < total) {
                task = t;
                PFaiT<EXACT> f; f.A = q.A[t]; f.sth = q.sth[t]; f.dvm = q.dvm[t];
                hs.init_warm(f, dz_guess(q.guess[t]), q.trig[q.guess[t]]);
            } else task = total;                     // queue drained for this lane
        }
        const bool active = task < total;
        if (!__any_sync(0xffffffffu, active)) break;
        if (active && hs.step()) { q.alpha[task] = hs.x; task = -1; }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// back half of step(): exchange, distance, terminal checks, danger zone, reward, observation, statistics
// partials, auto-reset. environment.py:130-179 / :212-255, :317-343, :346-396.
// FUSED = true: front half in the same kernel (cw mode, where propagation is one 6x6 product).
// STARTS = true (auto_reset == SAT_RESET_STARTS): a reset puts the env at its start columns (SAT_COL_START..+11) with
// int_state = 0 instead of at reset_p / reset_e with int_state = 1. The two lanes of an env agree on reset_now but the
// lanes of a warp do not, so nothing in the reset branches exchanges across lanes: each lane loads the columns it needs.
// ---------------------------------------------------------------------------------------------
template <bool FUSED, typename ActT, int MINB, bool EXACT, bool STARTS = false>
__global__ void __launch_bounds__(kBlock, MINB)
env_step_kernel(const SatEnvState st, const ActT* __restrict__ pa, const ActT* __restrict__ ea,
                const int32_t* __restrict__ count_override, float* __restrict__ obs_f32,
                double* __restrict__ obs_f64, double* __restrict__ term_obs_f64,
                double* __restrict__ reward_out, uint8_t* __restrict__ done_out,
                const double* __restrict__ dis_prev_in, double* __restrict__ partials,
                unsigned int* __restrict__ ticket, const __grid_constant__ SatEnvParams p) {
    // the solve queue and the pre-reset observation tile are live at different times: one shared-memory block, two views
    union SharedBlock { SolveQueue queue; double tile_term[kEnvsPerBlock][kObs]; __device__ SharedBlock() {} };
    __shared__ SharedBlock shm;
    __shared__ double tile[kEnvsPerBlock][kStatDims];               // next observation (+ return) of the CTA's envs
    SolveQueue& queue = shm.queue;
    double (&tile_term)[kEnvsPerBlock][kObs] = shm.tile_term;       // pre-reset observation
    queue_init<EXACT>(queue);

    const int64_t tid = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    const int64_t env_raw = tid >> 1;
    const int craft = (int)(tid & 1);
    const bool valid = env_raw < st.n;
    const int64_t e = valid ? env_raw : st.n - 1;
    const int64_t ld = st.ld;
    double* __restrict__ S = st.state;
    int32_t* __restrict__ I = st.istate;
    if (ticket && blockIdx.x == 0 && threadIdx.x == 0) *ticket = 0u;   // consumed by stats_merge_kernel (next in stream)

    Lane L;
    load_and_gate(st, p, pa, ea, e, craft, L, FUSED);
    if (FUSED) propagate_cw(p, L);
    else L.dis_prev = dis_prev_in[e];
    const int dz_stale = I[SAT_ICOL_DZ * ld + e];
    const int count = I[SAT_ICOL_COUNT * ld + e];
    int err = I[SAT_ICOL_ERR * ld + e];
    const double ret = S[SAT_COL_RET * ld + e];

    // ---------------- exchange, distance, terminal checks (:130-147)
    double P[3], Pv[3], E[3], Ev[3], d[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double o_r = shfl1(L.r[k]), o_v = shfl1(L.v[k]);
        P[k] = craft == 0 ? L.r[k] : o_r;  Pv[k] = craft == 0 ? L.v[k] : o_v;
        E[k] = craft == 0 ? o_r : L.r[k];  Ev[k] = craft == 0 ? o_v : L.v[k];
        d[k] = __dsub_rn(P[k], E[k]);
    }
    const double dis = norm3(d);                                              // :132
    const int count_new = count_override ? count_override[e] : count + 1;
    const bool captured = dis <= p.d_capture;                                 // :139
    const bool timeout = count_new >= p.max_episode_steps;                    // :144
    const bool done = captured || timeout;
    const double fuel_oth = shfl1(L.fuel_own);
    const double fuel_c = craft == 0 ? L.fuel_own : fuel_oth;                 // Delta_V_c = fuel_c (:328)
    double pa_gated[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { const double o = shfl1(L.a[k]); pa_gated[k] = craft == 0 ? L.a[k] : o; }

    // ---------------- next observation (after the auto reset, environment.py:66-79): it depends on the propagated state
    // and the terminal checks only, so it is stored BEFORE the danger-zone solve (88 % of the step's output bytes leave
    // early; measured neutral on both the device-resident and the host-buffer path, and it frees 12 registers' worth of
    // spills because P/E/Pv/Ev need not stay live across the solve for the observation)
    const int le = threadIdx.x >> 1;       // env slot within the CTA
    const bool reset_now = done && p.auto_reset;
    const int64_t env0 = (int64_t)blockIdx.x * kEnvsPerBlock;
    const int64_t rem = st.n - env0;
    const int rows = (int)(rem < kEnvsPerBlock ? rem : kEnvsPerBlock);
    {
        double Po[3], Pvo[3], Eo[3], Evo[3];
        if (STARTS) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { Po[k] = P[k]; Pvo[k] = Pv[k]; Eo[k] = E[k]; Evo[k] = Ev[k]; }
            if (reset_now) {
                const double* __restrict__ Sst = S + SAT_COL_START * ld;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    Po[k] = Sst[(SAT_COL_P + k) * ld + e];  Pvo[k] = Sst[(SAT_COL_PV + k) * ld + e];
                    Eo[k] = Sst[(SAT_COL_E + k) * ld + e];  Evo[k] = Sst[(SAT_COL_EV + k) * ld + e];
                }
            }
        } else {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                Po[k] = reset_now ? p.reset_p[k] : P[k];  Pvo[k] = reset_now ? 0.0 : Pv[k];
                Eo[k] = reset_now ? p.reset_e[k] : E[k];  Evo[k] = reset_now ? 0.0 : Ev[k];
            }
        }
        if (craft == 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { tile[le][k] = __dsub_rn(Po[k], Eo[k]); tile[le][3 + k] = __dsub_rn(Pvo[k], Evo[k]); tile[le][6 + k] = Po[k]; }
        } else {
#pragma unroll
            for (int k = 0; k < 3; ++k) { tile[le][9 + k] = Pvo[k]; tile[le][12 + k] = Eo[k]; tile[le][15 + k] = Evo[k]; }
        }
        __syncthreads();
        const int total = rows * kObs;
        for (int idx = threadIdx.x; idx < total; idx += kBlock) {
            const int row = idx / kObs, col = idx - row * kObs;
            const double val = tile[row][col];
            if (obs_f32) obs_f32[env0 * kObs + idx] = (float)val;
            if (obs_f64) obs_f64[env0 * kObs + idx] = val;
        }
    }

    // ---------------- danger-zone count (:150 -> :317-332), three phases with CTA-wide solve compaction
    // Flag 2 (environment.py:257-298, the dynamics in front of the surrogate training): no danger-zone evaluation, reward 0
    const bool need_dz = !done && !p.skip_danger_zone && p.flag != 2;
    DzNode nd;
    {
        double Ri[3], Vi[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) { Ri[k] = __dadd_rn(p.r_cw[k], L.r[k]); Vi[k] = __dadd_rn(p.v_cw[k], L.v[k]); }   // :338-341
        dz_prepare<EXACT>(craft, need_dz, Ri, Vi, fuel_c, p.u_grav, nd);
    }
    int slot0, slot1;
    double alpha0, alpha1;
    queue_push(queue, nd, slot0, slot1, alpha0, alpha1);
    queue_run<EXACT>(queue);
    if (slot0 >= 0) alpha0 = queue.alpha[slot0];
    if (slot1 >= 0) alpha1 = queue.alpha[slot1];
    __syncthreads();                                        // queue storage is reused by the observation tiles below
    const int dz_eval = dz_finalize<EXACT>(need_dz, nd, alpha0, alpha1, nullptr);
    int dz_new = dz_stale;                                   // not refreshed on capture / time-out steps (Q3)
    if (need_dz) {
        if (dz_eval >= 0) dz_new = dz_eval;
        else { dz_new = 0; err = 1; }        // the reference raises here (circular / parabolic element set)
    }

    // ---------------- reward (:139-147, :161-175, Flag 1 :221-251)
    double reward = 0.0, cos_a = 0.0, cos_b = 0.0;
    if (p.flag == 2) reward = 0.0;                                                            // :303-316
    else if (captured) reward = (p.flag == 0) ? 100.0 : -150.0;
    else if (timeout) reward = (p.flag == 0) ? 0.0 : 100.0;
    else {
        // the four cosines are split over the lane pair (2 each) and swapped: same values, half the latency. The operands
        // are SELECTED per lane and both lanes run the same two cosine3 calls - a branch on `craft` would make every warp
        // execute all four with half its lanes masked.
        const bool pv4_on = pa_gated[0] != 0.0 && pa_gated[1] != 0.0 && pa_gated[2] != 0.0;       // :169, else pv4 = 0
        double u1[3], w1[3], u2[3], w2[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            u1[k] = craft == 0 ? P[k] : d[k];   w1[k] = craft == 0 ? E[k] : Pv[k];               // pv1 :166 | pv3 :168
            u2[k] = craft == 0 ? Pv[k] : d[k];  w2[k] = craft == 0 ? Ev[k] : (pv4_on ? pa_gated[k] : Pv[k]);   // pv2 :167 | pv4 :169
        }
        const double ca = cosine3(u1, w1);
        double cb = cosine3(u2, w2);
        if (craft == 1) cb = pv4_on ? -cb : 0.0;
        cos_a = ca; cos_b = cb;
    }
    // (warp-convergent point: the swaps below are executed by every lane)
    const double oth_a = shfl1(cos_a), oth_b = shfl1(cos_b);
    if (!captured && !timeout && p.flag != 2) {
        const double pv1 = craft == 0 ? cos_a : oth_a, pv2 = craft == 0 ? cos_b : oth_b;
        const double pv3 = craft == 0 ? oth_a : cos_a, pv4 = craft == 0 ? oth_b : cos_b;
        const double ra = (dis < L.dis_prev) ? 1.0 : -1.0;                                    // :161
        const double rb = (p.d_capture <= dis && dis <= 4.0 * p.d_capture) ? -1.0 : -2.0;     // :162
        const double rc = (dz_new == 0) ? -1.0 : dz_new * 0.5;                                // :164
        double rr = __dadd_rn(__dadd_rn(ra, rb), rc);
        rr = __dadd_rn(rr, pv1);                                                              // :172-175
        rr = __dadd_rn(rr, __dmul_rn(0.6, pv2));
        rr = __dadd_rn(rr, __dmul_rn(0.2, pv3));
        rr = __dadd_rn(rr, __dmul_rn(2.0, pv4));
        reward = (p.flag == 0) ? rr : -rr;                                                    // :251
    }
    // discounted return of RewardScaling (normalization.py:57), reset on done (:62-63)
    const double ret_new = __dadd_rn(__dmul_rn(p.gamma, ret), reward);

    // ---------------- observation before reset (what the reference returns as s_)
    if (term_obs_f64) {
        if (craft == 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { tile_term[le][k] = d[k]; tile_term[le][3 + k] = __dsub_rn(Pv[k], Ev[k]); tile_term[le][6 + k] = P[k]; }
        } else {
#pragma unroll
            for (int k = 0; k < 3; ++k) { tile_term[le][9 + k] = Pv[k]; tile_term[le][12 + k] = E[k]; tile_term[le][15 + k] = Ev[k]; }
        }
    }

    // ---------------- auto reset (environment.py:66-79; fuel/dis/dangerous_zone persist, Q2)
    int int_state_new = 0, count_store = count_new;
    if (STARTS) {
        // reset to the env's start: the lane's own craft from the start columns (re-read rather than kept live across
        // the danger-zone solve). Starts are floats, so no int64 truncation follows (int_state = 0).
        if (reset_now) {
            const double* __restrict__ Sst = S + (SAT_COL_START + craft * 6) * ld;
#pragma unroll
            for (int k = 0; k < 3; ++k) { L.r[k] = Sst[k * ld + e]; L.v[k] = Sst[(3 + k) * ld + e]; }
            count_store = 0;
        }
    } else if (reset_now) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            P[k] = p.reset_p[k]; E[k] = p.reset_e[k]; Pv[k] = 0.0; Ev[k] = 0.0;
            L.r[k] = craft == 0 ? P[k] : E[k]; L.v[k] = 0.0;
        }
        int_state_new = 1; count_store = 0;
    }

    // ---------------- store state
    if (valid) {
        const int base = craft * 6;
        if (FUSED || reset_now) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { S[(base + k) * ld + e] = L.r[k]; S[(base + 3 + k) * ld + e] = L.v[k]; }
        }
        if (FUSED) S[(SAT_COL_FUEL_C + craft) * ld + e] = L.fuel_own;
        if (craft == 0) {
            S[SAT_COL_DIS * ld + e] = dis;
            S[SAT_COL_RET * ld + e] = done ? 0.0 : ret_new;
            I[SAT_ICOL_DZ * ld + e] = dz_new;
            I[SAT_ICOL_COUNT * ld + e] = count_store;
            reward_out[e] = reward;
            done_out[e] = done ? 1 : 0;
        } else {
            I[SAT_ICOL_INTSTATE * ld + e] = int_state_new;
            I[SAT_ICOL_ERR * ld + e] = err;
        }
    }

    // ---------------- pre-reset observation stores + per-CTA statistics partial (the tile holds the next observation)
    if (craft == 0) tile[le][18] = ret_new;
    __syncthreads();
    if (term_obs_f64) {
        const int total = rows * kObs;
        for (int idx = threadIdx.x; idx < total; idx += kBlock) {
            const int row = idx / kObs, col = idx - row * kObs;
            term_obs_f64[env0 * kObs + idx] = tile_term[row][col];
        }
    }
    if (partials && threadIdx.x < kStatDims) {
        // two-pass mean / M2 over the CTA's rows in a fixed order (deterministic)
        const int dim = threadIdx.x;
        double sum = 0.0;
        for (int row = 0; row < rows; ++row) sum += tile[row][dim];
        const double mean = sum / rows;
        double m2 = 0.0;
        for (int row = 0; row < rows; ++row) { double t = tile[row][dim] - mean; m2 += t * t; }
        partials[((int64_t)blockIdx.x * kStatDims + dim) * 2 + 0] = mean;
        partials[((int64_t)blockIdx.x * kStatDims + dim) * 2 + 1] = m2;
    }
}

// ---------------------------------------------------------------------------------------------
// batched danger-zone count on explicit inertial states (Time_window_of_danger_zone(...)
// .calculate_number_of_hanger_area(), satellite_function.py:18-99, 341-373)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
danger_zone_kernel(const double* __restrict__ rv, const double* __restrict__ dv, int64_t n, double u_grav,
                   int32_t* __restrict__ count_out, double* __restrict__ debug_out) {
    __shared__ SolveQueue queue;
    queue_init(queue);
    const int64_t tid = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    const int64_t env_raw = tid >> 1;
    const int craft = (int)(tid & 1);
    const bool valid = env_raw < n;
    const int64_t e = valid ? env_raw : n - 1;
    double Ri[3], Vi[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { Ri[k] = rv[e * 12 + craft * 6 + k]; Vi[k] = rv[e * 12 + craft * 6 + 3 + k]; }
    DzNode nd;
    dz_prepare(craft, true, Ri, Vi, dv[e], u_grav, nd);
    int slot0, slot1;
    double alpha0, alpha1;
    queue_push(queue, nd, slot0, slot1, alpha0, alpha1);
    queue_run(queue);
    if (slot0 >= 0) alpha0 = queue.alpha[slot0];
    if (slot1 >= 0) alpha1 = queue.alpha[slot1];
    DzDebug dbg = {0, 0, 0, 0, 0, 0, 0, 0};
    const int dz = dz_finalize(true, nd, alpha0, alpha1, debug_out ? &dbg : nullptr);
    if (valid) {
        if (craft == 0) count_out[e] = dz;
        if (debug_out) {
            double* o = debug_out + (e * 2 + craft) * 8;
            o[0] = dbg.rf_max; o[1] = dbg.rf_min; o[2] = dbg.r_ft; o[3] = dbg.alpha0; o[4] = dbg.alpha1;
            o[5] = dbg.theta; o[6] = dbg.dvm; o[7] = dbg.f_cx;
        }
    }
}

// one fsolve per thread, straight-line form of the same Hybrd1<PFai> the env step runs (satellite_function.py:558-565)
__global__ void __launch_bounds__(kBlock)
fsolve_pfai_kernel(const double* __restrict__ dvm, const double* __restrict__ theta, const double* __restrict__ v1x,
                   const double* __restrict__ v1y, const double* __restrict__ h, const double* __restrict__ guess,
                   int64_t n, double u_grav, double* __restrict__ root_out, int32_t* __restrict__ nfev_out) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    double sth, cth;
    glibm::sincos(theta[i], &sth, &cth);
    PFai f;
    f.A = (2.0 * u_grav * (1.0 - cth)) / (h[i] * v1y[i]) - v1x[i] * sth / v1y[i];      // :560
    f.sth = sth;
    f.dvm = dvm[i];
    Hybrd1<PFai> hs;
    hs.init(f, guess[i]);
    while (!hs.step()) {}
    root_out[i] = hs.x;
    if (nfev_out) nfev_out[i] = hs.nfev;
}

__global__ void __launch_bounds__(256)
libm_eval_kernel(int fn, const double* __restrict__ x, double* __restrict__ y, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    double r = 0.0, s, c;
    switch (fn) {
        case SAT_LIBM_SIN: r = glibm::sin(v); break;
        case SAT_LIBM_COS: r = glibm::cos(v); break;
        case SAT_LIBM_ACOS: r = glibm::acos(v); break;
        case SAT_LIBM_ATAN: r = glibm::atan(v); break;
        case SAT_LIBM_POW2: r = glibm::pow2(v); break;
        case SAT_LIBM_SINCOS_S: glibm::sincos(v, &s, &c); r = s; break;
        default: glibm::sincos(v, &s, &c); r = c; break;
    }
    y[i] = r;
}

// ---------------------------------------------------------------------------------------------
// merge of per-CTA partials into the running statistics (RunningMeanStd, normalization.py:19-29).
// One CTA per statistic dimension; two-pass (grand mean, then M2 about it) with fixed summation order ->
// bitwise deterministic. The last CTA to finish (ticket) advances the sample counts.
// ---------------------------------------------------------------------------------------------
struct Moments { double n, mean, m2; };
SAT_DEV Moments chan(Moments A, Moments B) {
    if (B.n == 0.0) return A;
    if (A.n == 0.0) return B;
    Moments C;
    C.n = A.n + B.n;
    const double delta = B.mean - A.mean;
    C.mean = A.mean + delta * (B.n / C.n);
    C.m2 = A.m2 + B.m2 + delta * delta * (A.n * B.n / C.n);
    return C;
}

SAT_DEV void fold_into_running(double* stats, int dim, int d, Moments B, double* std_out) {
    // stats: [0]=n, mean[dim], S[dim], std[dim]
    const double n_old = stats[0];
    const double mean_old = stats[1 + d], S_old = stats[1 + dim + d];
    double n_new, mean_new, S_new, std_new;
    if (B.n == 1.0) {
        // literal Welford step of the reference incl. its first-sample rule (normalization.py:21-29)
        const double x = B.mean;
        n_new = n_old + 1.0;
        if (n_new == 1.0) { mean_new = x; S_new = S_old; std_new = x; }
        else {
            mean_new = mean_old + (x - mean_old) / n_new;
            S_new = S_old + (x - mean_old) * (x - mean_new);
            std_new = sqrt(S_new / n_new);
        }
    } else {
        Moments A = {n_old, mean_old, S_old};
        Moments C = chan(A, B);
        n_new = C.n; mean_new = C.mean; S_new = C.m2;
        std_new = sqrt(S_new / n_new);
    }
    stats[1 + d] = mean_new; stats[1 + dim + d] = S_new; stats[1 + 2 * dim + d] = std_new;
    if (std_out) *std_out = std_new;
}

constexpr int kMergeThreads = 256;

SAT_DEV double block_sum_fixed(double v, double* sm) {
    // warp tree (xor) then the per-warp sums added in warp order by every thread: fixed order, all threads get the result
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kMergeThreads / 32; ++w) t += sm[w];
    return t;
}

// Per-CTA partials as the merge reads them: at(b, dim, nb) is the (mean, M2) pair of block b and sets nb to its row count;
// rewind() precedes each pass over b = threadIdx.x, threadIdx.x + kMergeThreads, ... (increasing).
// One batch: n_rows rows cut into blocks of rows_per_block.
struct OneBatch {
    const double* partials;
    int64_t n_rows;
    int rows_per_block, ndims;
    SAT_DEV void rewind() {}
    SAT_DEV const double* at(int64_t b, int dim, double& nb) {
        const int64_t rem = n_rows - b * rows_per_block;
        nb = (double)(rem < rows_per_block ? rem : rows_per_block);
        return partials + (b * ndims + dim) * 2;
    }
};

// The batches of G ranks, gathered rank-major with a stride of `stride` blocks per rank; rank r holds rank_rows[r] rows.
// Global block b runs over rank 0's blocks, then rank 1's, ...: the block order of the union batch whenever every rank
// but the last holds a multiple of rows_per_block rows.
struct RankMajor {
    const double* partials;
    const int64_t* rank_rows;
    int64_t stride;
    int rows_per_block, ndims;
    int r;
    int64_t b0, b1;                              // global blocks [b0, b1) are rank r's
    SAT_DEV int64_t blocks_of(int64_t rows) const { return (rows + rows_per_block - 1) / rows_per_block; }
    SAT_DEV void rewind() { r = 0; b0 = 0; b1 = blocks_of(rank_rows[0]); }
    SAT_DEV const double* at(int64_t b, int dim, double& nb) {
        while (b >= b1) { ++r; b0 = b1; b1 += blocks_of(rank_rows[r]); }
        const int64_t j = b - b0;
        const int64_t rem = rank_rows[r] - j * rows_per_block;
        nb = (double)(rem < rows_per_block ? rem : rows_per_block);
        return partials + ((r * stride + j) * ndims + dim) * 2;
    }
};

// pass 1: grand mean of the block means weighted by their rows; pass 2: M2 about it. Each thread sums its blocks in
// increasing b, then block_sum_fixed: the result depends only on the sequence of blocks.
template <class Blocks>
SAT_DEV void merge_fold(Blocks blocks, int64_t nblocks, double N, double* sm, double* obs_stats, int obs_dim,
                        double* ret_stats, double* ret_std_out, unsigned int* ticket) {
    const int dim = blockIdx.x;                  // gridDim.x == number of statistic dims in the partials
    double wsum = 0.0;
    blocks.rewind();
    for (int64_t b = threadIdx.x; b < nblocks; b += kMergeThreads) {
        double nb;
        const double* q = blocks.at(b, dim, nb);
        wsum += nb * q[0];
    }
    const double grand = block_sum_fixed(wsum, sm) / N;
    double m2 = 0.0;
    blocks.rewind();
    for (int64_t b = threadIdx.x; b < nblocks; b += kMergeThreads) {
        double nb;
        const double* q = blocks.at(b, dim, nb);
        const double dm = q[0] - grand;
        m2 += q[1] + nb * dm * dm;
    }
    m2 = block_sum_fixed(m2, sm);
    if (threadIdx.x == 0) {
        Moments B = {N, grand, m2};
        if (dim < obs_dim) { if (obs_stats) fold_into_running(obs_stats, obs_dim, dim, B, nullptr); }
        else if (ret_stats) fold_into_running(ret_stats, 1, 0, B, ret_std_out);
        __threadfence();
        const unsigned int t = atomicAdd(ticket, 1u);
        if (t == gridDim.x - 1) {                // every dimension has read the old counts: advance them
            if (obs_stats) obs_stats[0] += N;
            if (ret_stats) ret_stats[0] += N;
            *ticket = 0u;
        }
    }
}

__global__ void __launch_bounds__(kMergeThreads)
stats_merge_kernel(const double* __restrict__ partials, int64_t nblocks, int64_t n_rows, int rows_per_block,
                   int ndims_in_partials, double* obs_stats, int obs_dim, double* ret_stats, double* ret_std_out,
                   unsigned int* ticket) {
    __shared__ double sm[kMergeThreads / 32];
    merge_fold(OneBatch{partials, n_rows, rows_per_block, ndims_in_partials}, nblocks, (double)n_rows, sm, obs_stats,
               obs_dim, ret_stats, ret_std_out, ticket);
}

// stats_merge_kernel over the gathered partials of G ranks (RankMajor); with G == 1 it is the same fold
__global__ void __launch_bounds__(kMergeThreads)
stats_fold_ranks_kernel(const double* __restrict__ partials, int G, int64_t stride, const int64_t* __restrict__ rank_rows,
                        int rows_per_block, int ndims_in_partials, double* obs_stats, int obs_dim, double* ret_stats,
                        double* ret_std_out, unsigned int* ticket) {
    __shared__ double sm[kMergeThreads / 32];
    int64_t n_rows = 0, nblocks = 0;
    for (int r = 0; r < G; ++r) {
        const int64_t m = rank_rows[r];
        n_rows += m;
        nblocks += (m + rows_per_block - 1) / rows_per_block;
    }
    if (n_rows == 0) return;                     // nothing to fold; the ticket stays 0
    merge_fold(RankMajor{partials, rank_rows, stride, rows_per_block, ndims_in_partials, 0, 0, 0}, nblocks,
               (double)n_rows, sm, obs_stats, obs_dim, ret_stats, ret_std_out, ticket);
}

// ---------------------------------------------------------------------------------------------
// init / reset / observe
// ---------------------------------------------------------------------------------------------
__global__ void env_init_kernel(const SatEnvState st, double fuel_c, double fuel_t,
                                const __grid_constant__ SatEnvParams p, const uint8_t* __restrict__ mask, int full) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= st.n) return;
    if (mask && !mask[e]) return;
    const int64_t ld = st.ld;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        st.state[(SAT_COL_P + k) * ld + e] = p.reset_p[k];     // environment.py:67
        st.state[(SAT_COL_PV + k) * ld + e] = 0.0;             // :68
        st.state[(SAT_COL_E + k) * ld + e] = p.reset_e[k];     // :70
        st.state[(SAT_COL_EV + k) * ld + e] = 0.0;             // :71
    }
    st.istate[SAT_ICOL_INTSTATE * ld + e] = 1;                 // int64 arrays until the first step (Q1)
    st.istate[SAT_ICOL_COUNT * ld + e] = 0;
    if (full) {                                                // constructor, environment.py:41-44
        st.state[SAT_COL_FUEL_C * ld + e] = fuel_c;
        st.state[SAT_COL_FUEL_T * ld + e] = fuel_t;
        st.state[SAT_COL_DIS * ld + e] = INFINITY;
        st.state[SAT_COL_RET * ld + e] = 0.0;
        st.istate[SAT_ICOL_DZ * ld + e] = 0;
        st.istate[SAT_ICOL_ERR * ld + e] = 0;
    }
}

// ---------------------------------------------------------------------------------------------
// per-env start states (SAT_STATE_COLS_STARTS-column buffers): reset to the start columns, and the draw of the next starts
// ---------------------------------------------------------------------------------------------
// reset() to the start: kinematics from columns SAT_COL_START..+11, count = 0, int_state = 0; fuel / dis / dangerous_zone /
// the discounted return persist, as in env_init_kernel's reset form
__global__ void env_reset_starts_kernel(const SatEnvState st, const uint8_t* __restrict__ mask) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= st.n) return;
    if (mask && !mask[e]) return;
    const int64_t ld = st.ld;
#pragma unroll
    for (int c = 0; c < 12; ++c) st.state[c * ld + e] = st.state[(SAT_COL_START + c) * ld + e];
    st.istate[SAT_ICOL_INTSTATE * ld + e] = 0;
    st.istate[SAT_ICOL_COUNT * ld + e] = 0;
}

struct StartBox { double lo[12], hi[12]; };

// Uniform draw in the box, keyed by (seed, global env id, draw index) only, so that a sharded batch and a resumed run
// draw the same starts. Philox4x32-10 with key (seed_lo, seed_hi ^ "SCN1") - never the actor noise's key for the same
// seed - and counter (g_lo, g_hi, draw, j): block j gives columns 2j (from c0:c1) and 2j + 1 (from c2:c3), each a 53-bit
// uniform u in [0, 1). Value lo + (hi - lo) * u with each operation rounded (-fmad=false), capped at hi; lo where lo == hi.
__global__ void env_draw_starts_kernel(const SatEnvState st, const uint8_t* __restrict__ mask, const StartBox box,
                                       uint64_t seed, uint32_t draw, int64_t row_offset) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= st.n) return;
    if (mask && !mask[e]) return;
    const int64_t ld = st.ld;
    const uint64_t g = (uint64_t)(row_offset + e);
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ 0x53434E31u;
    double* __restrict__ out = st.state + SAT_COL_START * ld + e;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        uint32_t c[4] = {(uint32_t)g, (uint32_t)(g >> 32), draw, (uint32_t)j};
        philox4x32_10(c, k0, k1);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int col = 2 * j + h;
            const uint64_t bits = (((uint64_t)c[2 * h] << 32) | c[2 * h + 1]) >> 11;
            const double u = (double)bits * 0x1p-53;
            const double lo = box.lo[col], hi = box.hi[col];
            double v = __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), u));
            v = v > hi ? hi : v;
            out[col * ld] = lo < hi ? v : lo;
        }
    }
}

__global__ void env_observe_kernel(const SatEnvState st, float* __restrict__ obs_f32, double* __restrict__ obs_f64) {
    // one thread per (env, obs element): reads are column-coalesced per element class, writes fully coalesced
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= st.n * kObs) return;
    const int64_t e = idx / kObs;
    const int j = (int)(idx - e * kObs);
    const int64_t ld = st.ld;
    const int k = j % 3, g = j / 3;
    double val;
    if (g == 0) val = __dsub_rn(st.state[(SAT_COL_P + k) * ld + e], st.state[(SAT_COL_E + k) * ld + e]);
    else if (g == 1) val = __dsub_rn(st.state[(SAT_COL_PV + k) * ld + e], st.state[(SAT_COL_EV + k) * ld + e]);
    else val = st.state[((g - 2) * 3 + k) * ld + e];
    if (obs_f32) obs_f32[idx] = (float)val;
    if (obs_f64) obs_f64[idx] = val;
}


// fp32 (normalised) observation for the policy networks: one thread per env reads its 12 state columns (coalesced over the
// envs), the 18 values go through a shared-memory tile and leave as full rows. Same arithmetic as env_observe_kernel.
constexpr int kObsNormEnvs = 128;
__global__ void __launch_bounds__(kObsNormEnvs)
env_observe_norm_kernel(const SatEnvState st, const double* __restrict__ obs_stats, float* __restrict__ obs_f32) {
    __shared__ float tile[kObsNormEnvs * kObs];
    const int64_t e0 = (int64_t)blockIdx.x * kObsNormEnvs;
    const int64_t e = e0 + threadIdx.x;
    const int64_t ld = st.ld;
    if (e < st.n) {
        double P[3], Pv[3], E[3], Ev[3], o[kObs];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            P[k] = st.state[(SAT_COL_P + k) * ld + e]; Pv[k] = st.state[(SAT_COL_PV + k) * ld + e];
            E[k] = st.state[(SAT_COL_E + k) * ld + e]; Ev[k] = st.state[(SAT_COL_EV + k) * ld + e];
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            o[k] = __dsub_rn(P[k], E[k]); o[3 + k] = __dsub_rn(Pv[k], Ev[k]);
            o[6 + k] = P[k]; o[9 + k] = Pv[k]; o[12 + k] = E[k]; o[15 + k] = Ev[k];
        }
#pragma unroll
        for (int j = 0; j < kObs; ++j) {
            double v = o[j];
            if (obs_stats) v = (v - obs_stats[1 + j]) / (obs_stats[1 + 2 * kObs + j] + 1e-8);
            tile[threadIdx.x * kObs + j] = (float)v;
        }
    }
    __syncthreads();
    const int64_t rem = st.n - e0;
    const int total = (int)(rem < kObsNormEnvs ? rem : kObsNormEnvs) * kObs;
    for (int idx = threadIdx.x; idx < total; idx += kObsNormEnvs) obs_f32[e0 * kObs + idx] = tile[idx];
}

// ---------------------------------------------------------------------------------------------
// stand-alone batch normalisation (Normalization.__call__, normalization.py:37-43)
// ---------------------------------------------------------------------------------------------
constexpr int kNormRows = 128;

__global__ void __launch_bounds__(kNormRows)
norm_partial_kernel(const double* __restrict__ x, int64_t n, int dim, double* __restrict__ partials,
                    unsigned int* __restrict__ ticket) {
    __shared__ double tile[kNormRows * 32];
    if (blockIdx.x == 0 && threadIdx.x == 0) *ticket = 0u;
    const int64_t row0 = (int64_t)blockIdx.x * kNormRows;
    const int64_t rem = n - row0;
    const int rows = (int)(rem < kNormRows ? rem : kNormRows);
    const int total = rows * dim;
    for (int idx = threadIdx.x; idx < total; idx += kNormRows) tile[idx] = x[row0 * dim + idx];
    __syncthreads();
    if (threadIdx.x < dim) {
        const int d = threadIdx.x;
        double sum = 0.0;
        for (int r = 0; r < rows; ++r) sum += tile[r * dim + d];
        const double mean = sum / rows;
        double m2 = 0.0;
        for (int r = 0; r < rows; ++r) { double t = tile[r * dim + d] - mean; m2 += t * t; }
        partials[((int64_t)blockIdx.x * dim + d) * 2 + 0] = mean;
        partials[((int64_t)blockIdx.x * dim + d) * 2 + 1] = m2;
    }
}

__global__ void norm_apply_kernel(const double* __restrict__ stats, const double* __restrict__ x, int64_t total,
                                  int dim, double* __restrict__ out64, float* __restrict__ out32) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int d = (int)(idx % dim);
    const double mean = stats[1 + d], sd = stats[1 + 2 * dim + d];
    const double y = (x[idx] - mean) / (sd + 1e-8);             // normalization.py:41
    if (out64) out64[idx] = y;
    if (out32) out32[idx] = (float)y;
}

int check_state(const SatEnvState* st) {
    if (!st || !st->state || !st->istate) return SAT_ERR_NULL;
    if (st->n <= 0 || st->ld < st->n || (st->ld & 1)) return SAT_ERR_SIZE;
    if (((uintptr_t)st->state & 15) || ((uintptr_t)st->istate & 15)) return SAT_ERR_SIZE;
    return SAT_OK;
}

inline int launch_status() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? SAT_OK : (int)e;
}

}  // namespace

extern "C" {

int64_t sat_workspace_bytes(int64_t n) {
    if (n <= 0) return kWsHeader;
    int64_t nb_env = (n + kEnvsPerBlock - 1) / kEnvsPerBlock;
    int64_t nb_norm = (n + kNormRows - 1) / kNormRows;
    int64_t a = nb_env * kStatDims * 2 * (int64_t)sizeof(double);
    int64_t b = nb_norm * 32 * 2 * (int64_t)sizeof(double);
    return ws_partials_offset(n) + (a > b ? a : b);
}

void sat_env_default_params(SatEnvParams* p) {
    if (!p) return;
    SatEnvParams q = {};
    q.mode = SAT_MODE_CW; q.flag = 0; q.max_episode_steps = 1000; q.auto_reset = 1;
    q.action_dtype = SAT_ACT_F32; q.substeps = 100; q.skip_danger_zone = 0;
    q.d_capture = 100000.0; q.d_range = 100000.0;                 // environment.py:28
    q.gamma = 0.99;                                               // CPPO_main.py:24
    q.h = 1.0; q.mu = 3.986e14; q.re = 6378137.0; q.j2 = 0.00108263;
    q.r_cw[0] = 27098000.0; q.r_cw[1] = 32306000.0; q.r_cw[2] = 0.0;   // environment.py:338
    q.v_cw[0] = -2350.0; q.v_cw[1] = 1970.0; q.v_cw[2] = 0.0;          // :339
    q.u_grav = 3.986e14;                                          // satellite_function.py:28
    q.reset_p[0] = 200000.0; q.reset_e[0] = 18000.0;              // environment.py:67,70
    *p = q;
}

int sat_env_init(const SatEnvState* st, double fuel_c, double fuel_t, const SatEnvParams* p, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!p) return SAT_ERR_NULL;
    const int threads = 256;
    const unsigned blocks = (unsigned)((st->n + threads - 1) / threads);
    env_init_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(*st, fuel_c, fuel_t, *p, nullptr, 1);
    return launch_status();
}

int sat_env_reset(const SatEnvState* st, const uint8_t* mask, const SatEnvParams* p, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!p) return SAT_ERR_NULL;
    const int threads = 256;
    const unsigned blocks = (unsigned)((st->n + threads - 1) / threads);
    env_init_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(*st, 0.0, 0.0, *p, mask, 0);
    return launch_status();
}

int sat_env_draw_starts(const SatEnvState* st, const uint8_t* mask, const double* lo_host, const double* hi_host,
                        uint64_t seed, uint32_t draw, int64_t row_offset, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!lo_host || !hi_host) return SAT_ERR_NULL;
    if (row_offset < 0) return SAT_ERR_SIZE;
    StartBox box;
    for (int c = 0; c < 12; ++c) {
        const double lo = lo_host[c], hi = hi_host[c];
        if (!std::isfinite(lo) || !std::isfinite(hi) || !(lo <= hi) || !std::isfinite(hi - lo)) return SAT_ERR_SIZE;
        box.lo[c] = lo; box.hi[c] = hi;
    }
    const int threads = 256;
    const unsigned blocks = (unsigned)((st->n + threads - 1) / threads);
    env_draw_starts_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(*st, mask, box, seed, draw, row_offset);
    return launch_status();
}

int sat_env_reset_starts(const SatEnvState* st, const uint8_t* mask, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    const int threads = 256;
    const unsigned blocks = (unsigned)((st->n + threads - 1) / threads);
    env_reset_starts_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(*st, mask);
    return launch_status();
}

int sat_env_observe_norm(const SatEnvState* st, const double* obs_stats, float* obs_f32, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!obs_f32) return SAT_ERR_NULL;
    const unsigned blocks = (unsigned)((st->n + kObsNormEnvs - 1) / kObsNormEnvs);
    env_observe_norm_kernel<<<blocks, kObsNormEnvs, 0, (cudaStream_t)stream>>>(*st, obs_stats, obs_f32);
    return launch_status();
}

int sat_env_observe(const SatEnvState* st, float* obs_f32, double* obs_f64, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!obs_f32 && !obs_f64) return SAT_ERR_NULL;
    const int threads = 256;
    const int64_t total = st->n * kObs;
    const unsigned blocks = (unsigned)((total + threads - 1) / threads);
    env_observe_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(*st, obs_f32, obs_f64);
    return launch_status();
}

}  // extern "C"

namespace {
// ev (nullable): 4 events recorded before the first launch and after the front / finish / merge launches.
// partials_out (nullable): the finish kernel's per-CTA statistics partials go there and are not merged.
int env_step_impl(const SatEnvState* st, const void* pa, const void* ea, const int32_t* count_override,
                  float* obs_f32, double* obs_f64, double* term_obs_f64, double* reward, uint8_t* done,
                  double* obs_stats, double* ret_stats, double* ret_std_out, void* workspace,
                  const SatEnvParams* p, void* stream, cudaEvent_t* ev, float* obs_early = nullptr,
                  cudaEvent_t front_done = nullptr, float* pa_copy = nullptr, float* ea_copy = nullptr,
                  double* partials_out = nullptr) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!pa || !ea || !reward || !done || !p) return SAT_ERR_NULL;
    const bool want_stats = obs_stats || ret_stats || partials_out;
    if ((want_stats || p->mode == SAT_MODE_RK4) && !workspace) return SAT_ERR_NULL;
    if (p->mode != SAT_MODE_CW && p->mode != SAT_MODE_RK4) return SAT_ERR_MODE;
    if (p->action_dtype != SAT_ACT_F32 && p->action_dtype != SAT_ACT_F64) return SAT_ERR_MODE;
    if (p->flag < 0 || p->flag > 2) return SAT_ERR_MODE;
    if (p->mode == SAT_MODE_RK4 && p->substeps < 1) return SAT_ERR_SIZE;
    if (workspace && ((uintptr_t)workspace & 15)) return SAT_ERR_SIZE;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = st->n;
    const int64_t nblocks = (n + kEnvsPerBlock - 1) / kEnvsPerBlock;
    char* ws = (char*)workspace;
    unsigned int* ticket = ws ? (unsigned int*)ws : nullptr;
    double* dis_prev = ws ? (double*)(ws + ws_disprev_offset()) : nullptr;
    double* partials = partials_out ? partials_out : want_stats ? (double*)(ws + ws_partials_offset(n)) : nullptr;
    if (ev) cudaEventRecord(ev[0], s);
    // exact host-libm arithmetic in the danger-zone path (default) or libdevice (SatEnvParams.fast_libm); resets to the
    // reference's literals or (auto_reset == SAT_RESET_STARTS) to each env's start columns
    const bool starts = p->auto_reset == SAT_RESET_STARTS;
#define SAT_LAUNCH_FINISH(FUSED, T, ...)                                                                                   \
    do {                                                                                                                   \
        if (starts) {                                                                                                      \
            if (p->fast_libm) env_step_kernel<FUSED, T, kFinishMinBlocks, false, true><<<(unsigned)nblocks, kBlock, 0, s>>>(__VA_ARGS__); \
            else env_step_kernel<FUSED, T, kFinishMinBlocks, true, true><<<(unsigned)nblocks, kBlock, 0, s>>>(__VA_ARGS__); \
        } else {                                                                                                           \
            if (p->fast_libm) env_step_kernel<FUSED, T, kFinishMinBlocks, false><<<(unsigned)nblocks, kBlock, 0, s>>>(__VA_ARGS__); \
            else env_step_kernel<FUSED, T, kFinishMinBlocks, true><<<(unsigned)nblocks, kBlock, 0, s>>>(__VA_ARGS__);      \
        }                                                                                                                  \
    } while (0)
    if (p->mode == SAT_MODE_CW) {
        // one fused kernel: the propagation is a 6x6 product
        if (ev) cudaEventRecord(ev[1], s);
        if (p->action_dtype == SAT_ACT_F32)
            SAT_LAUNCH_FINISH(true, float, *st, (const float*)pa, (const float*)ea,
                count_override, obs_f32, obs_f64, term_obs_f64, reward, done, nullptr, partials, ticket, *p);
        else
            SAT_LAUNCH_FINISH(true, double, *st, (const double*)pa, (const double*)ea,
                count_override, obs_f32, obs_f64, term_obs_f64, reward, done, nullptr, partials, ticket, *p);
    } else {
        // kernel A (FP64-pipe bound, <= 72 registers, whole batch resident) then kernel B (register-heavy, divergent)
        const int64_t fblocks = (2 * n + kFrontBlock - 1) / kFrontBlock;
        if (obs_early && (count_override || p->action_dtype != SAT_ACT_F32 || !pa_copy || !ea_copy)) return SAT_ERR_MODE;
        if (obs_early) {
            if (starts)
                env_front_rk4_kernel<float, true, true><<<(unsigned)fblocks, kFrontBlock, 0, s>>>(
                    *st, (const float*)pa, (const float*)ea, dis_prev, obs_early, pa_copy, ea_copy, *p);
            else
                env_front_rk4_kernel<float, true><<<(unsigned)fblocks, kFrontBlock, 0, s>>>(*st, (const float*)pa, (const float*)ea,
                                                                                           dis_prev, obs_early, pa_copy, ea_copy, *p);
            if (front_done) cudaEventRecord(front_done, s);
            SAT_LAUNCH_FINISH(false, float, *st, pa_copy, ea_copy,
                count_override, obs_f32, obs_f64, term_obs_f64, reward, done, dis_prev, partials, ticket, *p);
        } else if (p->action_dtype == SAT_ACT_F32) {
            env_front_rk4_kernel<float, false><<<(unsigned)fblocks, kFrontBlock, 0, s>>>(*st, (const float*)pa, (const float*)ea, dis_prev, nullptr, nullptr, nullptr, *p);
            if (ev) cudaEventRecord(ev[1], s);
            SAT_LAUNCH_FINISH(false, float, *st, (const float*)pa, (const float*)ea,
                count_override, obs_f32, obs_f64, term_obs_f64, reward, done, dis_prev, partials, ticket, *p);
        } else {
            env_front_rk4_kernel<double, false><<<(unsigned)fblocks, kFrontBlock, 0, s>>>(*st, (const double*)pa, (const double*)ea, dis_prev, nullptr, nullptr, nullptr, *p);
            if (ev) cudaEventRecord(ev[1], s);
            SAT_LAUNCH_FINISH(false, double, *st, (const double*)pa, (const double*)ea,
                count_override, obs_f32, obs_f64, term_obs_f64, reward, done, dis_prev, partials, ticket, *p);
        }
    }
#undef SAT_LAUNCH_FINISH
    rc = launch_status();
    if (rc) return rc;
    if (ev) cudaEventRecord(ev[2], s);
    if (partials && !partials_out) {
        stats_merge_kernel<<<kStatDims, kMergeThreads, 0, s>>>(partials, nblocks, n, kEnvsPerBlock, kStatDims,
                                                               obs_stats, kObs, ret_stats, ret_std_out, ticket);
        rc = launch_status();
    }
    if (ev) cudaEventRecord(ev[3], s);
    return rc;
}

// d_io of sat_env_step_host: pa | ea (fp32 [n][3] each) | obs fp32 [n][18] | reward fp64 [n] | done u8 [n] | the env
// step's workspace, each region 256-byte aligned; `bytes` is the size of the whole buffer
struct HostIo {
    float *pa, *ea, *obs;
    double* reward;
    uint8_t* done;
    void* ws;
    int64_t bytes;
};
inline HostIo host_io_carve(void* d_io, int64_t n) {
    const uintptr_t base = (uintptr_t)d_io;
    int64_t off = 0;
    auto take = [&](int64_t b) { const uintptr_t p = base + (uintptr_t)off; off += (b + 255) / 256 * 256; return p; };
    HostIo io;
    io.pa = (float*)take(n * 12);
    io.ea = (float*)take(n * 12);
    io.obs = (float*)take(n * 72);
    io.reward = (double*)take(n * 8);
    io.done = (uint8_t*)take(n);
    io.ws = (void*)(base + (uintptr_t)off);
    io.bytes = off + sat_workspace_bytes(n);
    return io;
}
}  // namespace

extern "C" {

int sat_env_step(const SatEnvState* st, const void* pa, const void* ea, const int32_t* count_override,
                 float* obs_f32, double* obs_f64, double* term_obs_f64, double* reward, uint8_t* done,
                 double* obs_stats, double* ret_stats, double* ret_std_out, void* workspace,
                 const SatEnvParams* p, void* stream) {
    return env_step_impl(st, pa, ea, count_override, obs_f32, obs_f64, term_obs_f64, reward, done, obs_stats, ret_stats,
                         ret_std_out, workspace, p, stream, nullptr);
}

int sat_env_step_timed(const SatEnvState* st, const void* pa, const void* ea, const int32_t* count_override,
                       float* obs_f32, double* obs_f64, double* term_obs_f64, double* reward, uint8_t* done,
                       double* obs_stats, double* ret_stats, double* ret_std_out, void* workspace,
                       const SatEnvParams* p, void* stream, float* ms_out) {
    if (!ms_out) return SAT_ERR_NULL;
    cudaEvent_t ev[4];
    for (int i = 0; i < 4; ++i) {
        cudaError_t ce = cudaEventCreate(&ev[i]);
        if (ce != cudaSuccess) return (int)ce;
    }
    int rc = env_step_impl(st, pa, ea, count_override, obs_f32, obs_f64, term_obs_f64, reward, done, obs_stats, ret_stats,
                           ret_std_out, workspace, p, stream, ev);
    if (rc == SAT_OK) {
        cudaError_t ce = cudaEventSynchronize(ev[3]);
        if (ce != cudaSuccess) rc = (int)ce;
        else for (int i = 0; i < 3; ++i) cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]);
    }
    for (int i = 0; i < 4; ++i) cudaEventDestroy(ev[i]);
    return rc;
}

int sat_danger_zone_count(const double* rv, const double* dv, int64_t n, double u_grav, int32_t* count_out,
                          double* debug_out, void* stream) {
    if (!rv || !dv || !count_out) return SAT_ERR_NULL;
    if (n <= 0) return SAT_ERR_SIZE;
    const int64_t nblocks = (n + kEnvsPerBlock - 1) / kEnvsPerBlock;
    danger_zone_kernel<<<(unsigned)nblocks, kBlock, 0, (cudaStream_t)stream>>>(rv, dv, n, u_grav, count_out, debug_out);
    return launch_status();
}

int sat_fsolve_pfai(const double* dvm, const double* theta, const double* v1x, const double* v1y, const double* h,
                    const double* guess, int64_t n, double u_grav, double* root_out, int32_t* nfev_out, void* stream) {
    if (!dvm || !theta || !v1x || !v1y || !h || !guess || !root_out) return SAT_ERR_NULL;
    if (n <= 0) return SAT_ERR_SIZE;
    fsolve_pfai_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(
        dvm, theta, v1x, v1y, h, guess, n, u_grav, root_out, nfev_out);
    return launch_status();
}

int sat_libm_eval(int fn, const double* x, double* y, int64_t n, void* stream) {
    if (!x || !y) return SAT_ERR_NULL;
    if (n <= 0) return SAT_ERR_SIZE;
    if (fn < SAT_LIBM_SIN || fn > SAT_LIBM_SINCOS_C) return SAT_ERR_MODE;
    libm_eval_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(fn, x, y, n);
    return launch_status();
}

int64_t sat_env_step_host_bytes(int64_t n) { return n > 0 ? host_io_carve(nullptr, n).bytes : 0; }

int sat_env_step_host(const SatEnvState* st, const float* pa_host, const float* ea_host,
                      float* obs_host, double* reward_host, uint8_t* done_host, void* d_io,
                      const SatEnvParams* p, void* stream, void* aux_stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!pa_host || !ea_host || !obs_host || !reward_host || !done_host || !d_io || !p) return SAT_ERR_NULL;
    cudaStream_t s0 = (cudaStream_t)stream, s1 = (cudaStream_t)aux_stream;
    const int64_t n = st->n;
    const HostIo io = host_io_carve(d_io, n);
    SatEnvParams q = *p;
    q.action_dtype = SAT_ACT_F32;
    // pinned (UVA-mapped) host buffers can be handed to the kernels directly (zero-copy)
    cudaPointerAttributes at;
    bool mapped = true;
    const void* ptrs[5] = {pa_host, ea_host, obs_host, reward_host, done_host};
    void* dev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    for (int i = 0; i < 5 && mapped; ++i) {
        mapped = cudaPointerGetAttributes(&at, ptrs[i]) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer != nullptr;
        dev[i] = at.devicePointer;
    }
    cudaGetLastError();
    cudaError_t ce;
    if (mapped && s1 && q.mode == SAT_MODE_RK4) {
        // kernel A reads the actions from host memory (zero-copy), leaves a copy in device memory for kernel B and writes
        // the step's next observation (88 % of the output bytes) to device memory; a copy engine moves the observation to
        // the host on the second stream while kernel B (danger zone, reward) runs; kernel B writes reward / done straight
        // to host memory. Kernel B must not READ host memory here: PCIe read requests may not pass the copy's posted
        // writes, which stalled it by ~50 us. Measured at 65 536 envs: 241 us/step (all zero-copy: 287; staged: 333).
        static thread_local cudaEvent_t front_ev[64] = {};   // one event per device ordinal (events belong to a device)
        int devid = 0;
        if ((ce = cudaGetDevice(&devid)) != cudaSuccess) return (int)ce;
        if (devid < 0 || devid >= 64) return SAT_ERR_SIZE;
        cudaEvent_t& fe = front_ev[devid];
        if (!fe && (ce = cudaEventCreateWithFlags(&fe, cudaEventDisableTiming)) != cudaSuccess) return (int)ce;
        rc = env_step_impl(st, dev[0], dev[1], nullptr, nullptr, nullptr, nullptr, (double*)dev[3], (uint8_t*)dev[4],
                           nullptr, nullptr, nullptr, io.ws, &q, (void*)s0, nullptr, io.obs, fe, io.pa, io.ea);
        if (rc) return rc;
        if ((ce = cudaStreamWaitEvent(s1, fe, 0)) != cudaSuccess) return (int)ce;
        if ((ce = cudaMemcpyAsync(obs_host, io.obs, (size_t)n * 72, cudaMemcpyDeviceToHost, s1)) != cudaSuccess) return (int)ce;
        if ((ce = cudaStreamSynchronize(s0)) != cudaSuccess) return (int)ce;
        return (int)cudaStreamSynchronize(s1);
    }
    if (mapped) {
        // the action reads and the observation / reward / done stores cross PCIe from inside the kernels
        rc = sat_env_step(st, dev[0], dev[1], nullptr, (float*)dev[2], nullptr, nullptr, (double*)dev[3], (uint8_t*)dev[4],
                          nullptr, nullptr, nullptr, io.ws, &q, (void*)s0);
        if (rc) return rc;
        return (int)cudaStreamSynchronize(s0);
    }
    // pageable host memory: staged copies through d_io
    if ((ce = cudaMemcpyAsync(io.pa, pa_host, (size_t)n * 12, cudaMemcpyHostToDevice, s0)) != cudaSuccess) return (int)ce;
    if ((ce = cudaMemcpyAsync(io.ea, ea_host, (size_t)n * 12, cudaMemcpyHostToDevice, s0)) != cudaSuccess) return (int)ce;
    rc = sat_env_step(st, io.pa, io.ea, nullptr, io.obs, nullptr, nullptr, io.reward, io.done, nullptr, nullptr, nullptr, io.ws,
                      &q, (void*)s0);
    if (rc) return rc;
    if ((ce = cudaMemcpyAsync(obs_host, io.obs, (size_t)n * 72, cudaMemcpyDeviceToHost, s0)) != cudaSuccess) return (int)ce;
    if ((ce = cudaMemcpyAsync(reward_host, io.reward, (size_t)n * 8, cudaMemcpyDeviceToHost, s0)) != cudaSuccess) return (int)ce;
    if ((ce = cudaMemcpyAsync(done_host, io.done, (size_t)n, cudaMemcpyDeviceToHost, s0)) != cudaSuccess) return (int)ce;
    return (int)cudaStreamSynchronize(s0);
}

int64_t sat_stats_partials_bytes(int64_t n, int dim) {
    if (n <= 0 || dim < 0 || dim > 32) return 0;
    if (dim == 0) return (n + kEnvsPerBlock - 1) / kEnvsPerBlock * kStatDims * 2 * (int64_t)sizeof(double);
    return (n + kNormRows - 1) / kNormRows * dim * 2 * (int64_t)sizeof(double);
}

int sat_env_step_partials(const SatEnvState* st, const void* pa, const void* ea, const int32_t* count_override,
                          float* obs_f32, double* obs_f64, double* term_obs_f64, double* reward, uint8_t* done,
                          double* partials, void* workspace, const SatEnvParams* p, void* stream) {
    if (!partials) return SAT_ERR_NULL;
    return env_step_impl(st, pa, ea, count_override, obs_f32, obs_f64, term_obs_f64, reward, done, nullptr, nullptr,
                         nullptr, workspace, p, stream, nullptr, nullptr, nullptr, nullptr, nullptr, partials);
}

int sat_norm_partials(const double* x, int64_t n, int dim, double* partials, void* workspace, void* stream) {
    if (!x || !partials || !workspace) return SAT_ERR_NULL;
    if (n <= 0 || dim < 1 || dim > 32) return SAT_ERR_SIZE;
    const int64_t nblocks = (n + kNormRows - 1) / kNormRows;
    norm_partial_kernel<<<(unsigned)nblocks, kNormRows, 0, (cudaStream_t)stream>>>(x, n, dim, partials,
                                                                                   (unsigned int*)workspace);
    return launch_status();
}

int sat_stats_fold(const double* partials, int ranks, int64_t rank_stride_blocks, const int64_t* rank_rows, int dim,
                   double* obs_stats, double* ret_stats, double* ret_std_out, void* workspace, void* stream) {
    if (!partials || !rank_rows || !workspace) return SAT_ERR_NULL;
    if (ranks < 1 || rank_stride_blocks < 1 || dim < 0 || dim > 32) return SAT_ERR_SIZE;
    if (dim > 0 && (ret_stats || ret_std_out)) return SAT_ERR_SIZE;
    if (!obs_stats && !ret_stats) return SAT_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (dim == 0)
        stats_fold_ranks_kernel<<<kStatDims, kMergeThreads, 0, s>>>(partials, ranks, rank_stride_blocks, rank_rows,
                                                                    kEnvsPerBlock, kStatDims, obs_stats, kObs, ret_stats,
                                                                    ret_std_out, (unsigned int*)workspace);
    else
        stats_fold_ranks_kernel<<<dim, kMergeThreads, 0, s>>>(partials, ranks, rank_stride_blocks, rank_rows, kNormRows,
                                                              dim, obs_stats, dim, nullptr, nullptr,
                                                              (unsigned int*)workspace);
    return launch_status();
}

int sat_norm_update(double* stats, const double* x, int64_t n, int dim, int update,
                    double* x_out_f64, float* x_out_f32, void* workspace, void* stream) {
    if (!stats || !x) return SAT_ERR_NULL;
    if (n <= 0 || dim < 1 || dim > 32) return SAT_ERR_SIZE;
    if (update && !workspace) return SAT_ERR_NULL;
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    if (update) {
        const int64_t nblocks = (n + kNormRows - 1) / kNormRows;
        char* ws = (char*)workspace;
        double* partials = (double*)(ws + ws_partials_offset(n));
        norm_partial_kernel<<<(unsigned)nblocks, kNormRows, 0, s>>>(x, n, dim, partials, (unsigned int*)ws);
        if ((rc = launch_status())) return rc;
        stats_merge_kernel<<<dim, kMergeThreads, 0, s>>>(partials, nblocks, n, kNormRows, dim,
                                                         stats, dim, nullptr, nullptr, (unsigned int*)ws);
        if ((rc = launch_status())) return rc;
    }
    if (x_out_f64 || x_out_f32) {
        const int64_t total = n * dim;
        norm_apply_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(stats, x, total, dim, x_out_f64, x_out_f32);
        if ((rc = launch_status())) return rc;
    }
    return SAT_OK;
}

}  // extern "C"
