// sat_math.cuh -- device math for the satellite environment kernels (sm_100a).
//
// Two kinds of arithmetic live here and are deliberately kept apart:
//   (1) "exact" helpers that reproduce, bit for bit, the IEEE operations the reference's numpy /
//       OpenBLAS calls perform (ddot, dnrm2-as-sqrt(dot), dgemv, cross, scalar +-*/), written with
//       explicit __dmul_rn/__dadd_rn/__fma_rn so no compiler flag can re-associate or fuse them;
//   (2) the RK4 propagator core, written with explicit fma() for minimum FP64-pipe instruction
//       count (106 per RK4+J2 step), whose parity bar is 1e-9 relative, not bit identity.
// Translation units that include this file are compiled with -fmad=false, so every fused
// operation in the binary is one that is spelled fma() here.
//   (3) the transcendental calls of the danger-zone path (sin, cos, acos, atan, and python's `x ** 2` = pow(x, 2.0))
//       go through glibm.cuh, a restatement of the host libm the reference runs on, because the integer danger-zone
//       count depends on their last bit (DESIGN.md s3).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "glibm.cuh"

#define SAT_DEV __device__ __forceinline__

namespace sat {

constexpr double kPi = 3.141592653589793;
constexpr double kTwoPi = 2 * 3.141592653589793;   // python: 2 * np.pi (exact doubling)

// ------------------------------------------------------------------------------------------
// (1) exact helpers
// ------------------------------------------------------------------------------------------
// np.dot(a3, b3): OpenBLAS ddot tail loop, fma-accumulated left to right (see DESIGN.md)
SAT_DEV double dot3(const double a[3], const double b[3]) {
    double s = __dmul_rn(a[0], b[0]);
    s = __fma_rn(a[1], b[1], s);
    s = __fma_rn(a[2], b[2], s);
    return s;
}
// np.linalg.norm(a3) = sqrt(a.dot(a))
SAT_DEV double norm3(const double a[3]) { return __dsqrt_rn(dot3(a, a)); }

// np.cross(a, b): products and differences rounded separately
SAT_DEV void cross3(const double a[3], const double b[3], double c[3]) {
    c[0] = __dsub_rn(__dmul_rn(a[1], b[2]), __dmul_rn(a[2], b[1]));
    c[1] = __dsub_rn(__dmul_rn(a[2], b[0]), __dmul_rn(a[0], b[2]));
    c[2] = __dsub_rn(__dmul_rn(a[0], b[1]), __dmul_rn(a[1], b[0]));
}

// np.dot(M6x6, x6): OpenBLAS Haswell dgemv_t: 4-lane products, (p0+p2)+(p1+p3), then the 2-element
// tail as fma(m4, x4, m5*x5)   (satellite_function.py:778-779)
SAT_DEV double gemv6_row(const double* __restrict__ m, const double x[6]) {
    double p0 = __dmul_rn(m[0], x[0]), p1 = __dmul_rn(m[1], x[1]);
    double p2 = __dmul_rn(m[2], x[2]), p3 = __dmul_rn(m[3], x[3]);
    double head = __dadd_rn(__dadd_rn(p0, p2), __dadd_rn(p1, p3));
    double tail = __fma_rn(m[4], x[4], __dmul_rn(m[5], x[5]));
    return __dadd_rn(head, tail);
}

// cosine between two 3-vectors the way reward_of_action1/2/3/4 compute it (environment.py:351-353):
// each vector divided by its norm, then np.dot
SAT_DEV double cosine3(const double a[3], const double b[3]) {
    double na = norm3(a), nb = norm3(b);
    double ua[3], ub[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { ua[k] = __ddiv_rn(a[k], na); ub[k] = __ddiv_rn(b[k], nb); }
    return dot3(ua, ub);
}

// ------------------------------------------------------------------------------------------
// (2) RK4 two-body + J2 core (script "轨道外推-龙格库塔算法.py":15-40), Nystrom form of classical RK4.
//     Accelerations are carried divided by -mu; the step constants absorb -mu.
// ------------------------------------------------------------------------------------------
struct Rk4Consts {
    double h;      // h
    double hh;     // h/2
    double cx3;    // -mu h^2/4
    double cx4;    // -mu h^2/2
    double cx1;    // -mu h^2/6
    double cv;     // -mu h/6
    double cj;     // 1.5 J2 Re^2   (0 -> two-body)
};

SAT_DEV Rk4Consts make_rk4_consts(double h, double mu, double re, double j2) {
    Rk4Consts c;
    c.h = h; c.hh = 0.5 * h;
    c.cx3 = -mu * h * h * 0.25; c.cx4 = -mu * h * h * 0.5; c.cx1 = -mu * h * h / 6.0; c.cv = -mu * h / 6.0;
    c.cj = 1.5 * j2 * re * re;
    return c;
}

// 1/sqrt(x) to ~1 ulp: MUFU.RSQ64H seed (rel. err <= 2^-22.9) + one Halley step (cubic): 5 FP64 ops
SAT_DEV double rsqrt_halley(double x) {
    double y0;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(x));
    double yy = y0 * y0;
    double e = fma(-x, yy, 1.0);
    double p = fma(0.375, e, 0.5);
    double pe = p * e;
    return fma(y0, pe, y0);
}

// a(x)/(-mu): 19 FP64-pipe instructions with J2, 13 without
template <bool J2>
SAT_DEV void accel_scaled(double x, double y, double z, double cj, double& ax, double& ay, double& az) {
    double zz = z * z;
    double r2 = fma(x, x, fma(y, y, zz));
    double ri = rsqrt_halley(r2);
    double ri2 = ri * ri;
    double ri3 = ri2 * ri;
    if (J2) {
        double c = cj * ri2;            // 1.5 J2 Re^2 / r^2
        double q = zz * ri2;            // (z/r)^2
        double t1 = fma(-5.0, q, 1.0);  // 1 - 5 (z/r)^2
        double g = ri3 * c;             // 1.5 J2 Re^2 / r^5
        double kxy = fma(g, t1, ri3);   // r^-3 (1 + c (1 - 5 (z/r)^2))
        double kz = fma(2.0, g, kxy);   // r^-3 (1 + c (3 - 5 (z/r)^2))
        ax = kxy * x; ay = kxy * y; az = kz * z;
    } else {
        ax = ri3 * x; ay = ri3 * y; az = ri3 * z;
    }
}

template <bool J2>
SAT_DEV void rk4_step(double (&x)[3], double (&v)[3], const Rk4Consts& c) {
    double a1[3], a2[3], a3[3], a4[3], xa[3], xb[3], xs[3];
    accel_scaled<J2>(x[0], x[1], x[2], c.cj, a1[0], a1[1], a1[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) xa[k] = fma(c.hh, v[k], x[k]);            // x0 + h/2 v0
    accel_scaled<J2>(xa[0], xa[1], xa[2], c.cj, a2[0], a2[1], a2[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) xs[k] = fma(c.cx3, a1[k], xa[k]);         // + h^2/4 a1
    accel_scaled<J2>(xs[0], xs[1], xs[2], c.cj, a3[0], a3[1], a3[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) { xb[k] = fma(c.h, v[k], x[k]); xs[k] = fma(c.cx4, a2[k], xb[k]); }   // x0 + h v0 + h^2/2 a2
    accel_scaled<J2>(xs[0], xs[1], xs[2], c.cj, a4[0], a4[1], a4[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double t = a2[k] + a3[k];
        double s3 = a1[k] + t;
        x[k] = fma(c.cx1, s3, xb[k]);                                      // x0 + h v0 + h^2/6 (a1+a2+a3)
        double w = (s3 + t) + a4[k];
        v[k] = fma(c.cv, w, v[k]);                                         // v0 + h/6 (a1+2a2+2a3+a4)
    }
}

// ------------------------------------------------------------------------------------------
// The transcendental calls of the danger-zone path. EXACT = true (default): the host libm's own arithmetic (glibm.cuh) ->
// the reference's integer count, bit for bit. EXACT = false (SatEnvParams.fast_libm = 1): CUDA's libdevice and x*x, 1-2 ulp
// from the host libm: ~3e-5 of the counts differ from the reference (round-1 behaviour), 24 us faster per 65 536-env step.
// ------------------------------------------------------------------------------------------
template <bool EXACT>
struct Lm {
    static SAT_DEV double2 sincos(double x) {
        if (EXACT) return glibm::call::sincos(x);
        double s, c; ::sincos(x, &s, &c); return make_double2(s, c);
    }
    static SAT_DEV double2 sincos_inline(double x) {          // the solver's single evaluation site
        double s, c;
        if (EXACT) glibm::sincos(x, &s, &c); else ::sincos(x, &s, &c);
        return make_double2(s, c);
    }
    static SAT_DEV double cos(double x) { return EXACT ? glibm::call::cos(x) : ::cos(x); }
    static SAT_DEV double acos(double x) { return EXACT ? glibm::call::acos(x) : ::acos(x); }
    static SAT_DEV double atan(double x) { return EXACT ? glibm::call::atan(x) : ::atan(x); }
    static SAT_DEV double pow2(double x) { return EXACT ? glibm::call::pow2(x) : x * x; }
};

// ------------------------------------------------------------------------------------------
// orbital elements, satellite_function.py:161-255. The reference returns a list whose length gives the branch:
//   6: [a, e, i, omega, Omega, f]   energy != 0, e != 0 (elliptic or hyperbolic)
//   5: [p, i, omega, Omega, f]      energy == 0 (parabolic, :186-190, :247-253)
//   4: [a, i, u, Omega]             e == 0 (circular, :212, :223-227)
// ALL = false (the danger-zone path; the reference's danger-zone code raises on the last two): returns 6, or 0 for the
// parabolic / circular branches. ALL = true: returns the length and writes the list into el's fields in order.
// ------------------------------------------------------------------------------------------
struct Elements { double a, e, i, omega, Omega, f; };

template <bool EXACT = true, bool ALL = false>
SAT_DEV int orbital_elements(double miu, const double R0[3], const double V0[3], Elements& el) {
    double r_norm = norm3(R0), v_norm = norm3(V0);                       // :183-184
    double r_dot_v = dot3(R0, V0);                                       // :185
    double v2 = Lm<EXACT>::pow2(v_norm);                                     // v_norm ** 2 (:186, :193)
    double energy = 2.0 / r_norm - v2 / miu;                             // :186
    double c1 = v2 / miu - 1.0 / r_norm, c2 = r_dot_v / miu;             // :193
    double E[3], H[3], N[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) E[k] = c1 * R0[k] - c2 * V0[k];
    double e = norm3(E);                                                 // :194
    cross3(R0, V0, H);                                                   // :197
    double h = norm3(H);                                                 // :199
    N[0] = -H[1]; N[1] = H[0]; N[2] = 0.0;                               // :206 cross([0,0,1], H)
    double n = norm3(N);                                                 // :208
    if constexpr (!ALL) {
        if (energy == 0.0 || e == 0.0) return 0;
    }
    el.a = 1.0 / fabs(energy);                                           // :188
    el.e = e;
    el.i = Lm<EXACT>::acos(H[2] / h);                                               // :210
    double omega = (n != 0.0) ? Lm<EXACT>::acos(dot3(N, E) / n / e) : 0.0;          // :214-217
    if (E[2] < 0.0) omega = kTwoPi - omega;                              // :221
    el.omega = omega;
    double Omega = (n != 0.0) ? Lm<EXACT>::acos(N[0] / n) : 0.0;                    // :230-233
    if (N[1] < 0.0) Omega = kTwoPi - Omega;                              // :237
    el.Omega = Omega;
    double f = Lm<EXACT>::acos(dot3(E, R0) / e / r_norm);                           // :242
    if (r_dot_v < 0.0) f = kTwoPi - f;
    el.f = f;
    if constexpr (ALL) {
        // e == 0: the reference leaves omega and f at 0 (above they are acos of 0 / 0) and computes u instead (:223-227)
        if (e == 0.0) {
            el.omega = 0.0; el.f = 0.0;
            double u = Lm<EXACT>::acos(dot3(N, R0) / n / r_norm);                  // :225
            if (R0[2] < 0.0) u = kTwoPi - u;
            if (energy != 0.0) { el = {el.a, el.i, u, el.Omega, 0.0, 0.0}; return 4; }
        }
        if (energy == 0.0) { el = {Lm<EXACT>::pow2(h) / miu, el.i, el.omega, el.Omega, el.f, 0.0}; return 5; }   // p (:201)
    }
    return 6;
}

// ------------------------------------------------------------------------------------------
// scipy.optimize.fsolve(P_fai_equation, alpha_guess): MINPACK hybrd for n = 1 with scipy's defaults
// (SURVEY.md Appendix B). f(alpha) = A (dvm cos alpha) + sth (-dvm sin alpha), satellite_function.py:559-562.
// Returns the iterate un-polished, exactly like the reference uses result[0].
// ------------------------------------------------------------------------------------------
template <bool EXACT>
struct PFaiT {
    double A, sth, dvm;
    SAT_DEV double at(double s, double c) const { return A * (dvm * c) + sth * (-dvm * s); }   // given sin, cos of alpha
    SAT_DEV double operator()(double alpha) const {
        const double2 sc = Lm<EXACT>::sincos_inline(alpha);
        return at(sc.x, sc.y);
    }
};

using PFai = PFaiT<true>;

// The iteration is written as a state machine with ONE function-evaluation site per step(): lanes of a
// warp that are in different phases (initial value / forward-difference Jacobian / trial point) or even on
// different root problems still execute the expensive sincos together. The arithmetic and its order are
// exactly MINPACK's (Appendix B), so the iterates are bit-identical to the straight-line form.
template <class F>
struct Hybrd1 {
    F f;
    // a / b for a >= +0, b > 0 (b may be NaN): identical bits to the plain quotient, but a == 0 never reaches the divider
    static SAT_DEV double zdiv(double a, double b) {
        const double q = ((a == 0.0) ? 1.0 : a) / b;
        return (a == 0.0 && b == b) ? 0.0 : q;
    }
    double x, fv, fnorm, d, delta, xnorm, r, q, qtf, h, xt, p, pnorm;
    int nfev, iter, ncsuc, ncfail, nslow1, nslow2, phase;   // phase 0: f(x0), 1: f(x+h) (Jacobian), 2: f(xt) (trial)
    bool jeval;

    SAT_DEV void init(const F& fn, double x0) {
        f = fn; x = x0; fv = 0.0; fnorm = 0.0; d = 0.0; delta = 0.0; xnorm = 0.0; r = 0.0; q = 1.0; qtf = 0.0;
        h = 0.0; xt = x0; p = 0.0; pnorm = 0.0;
        nfev = 0; iter = 1; ncsuc = 0; ncfail = 0; nslow1 = 0; nslow2 = 0; phase = 0; jeval = true;
    }
    SAT_DEV void start_outer() {
        const double sqeps = 1.4901161193847656e-08;          // sqrt(machine eps), exact power of two
        h = sqeps * fabs(x);
        if (h == 0.0) h = sqeps;
        phase = 1;
    }
    SAT_DEV void dogleg() {
        const double epsmch = 2.220446049250313e-16;
        double t = r;
        if (t == 0.0) { t = epsmch * fabs(r); if (t == 0.0) t = epsmch; }
        const double xgn = qtf / t, qnorm = fabs(d * xgn);
        double step;
        if (qnorm <= delta) step = xgn;
        else {
            double w = (r * qtf) / d, gnorm = fabs(w), sgnorm = 0.0, alpha = delta / qnorm;
            if (gnorm != 0.0) {
                w = (w / gnorm) / d;
                const double tt = fabs(r * w);
                sgnorm = (gnorm / tt) / tt; alpha = 0.0;
                if (sgnorm < delta) {
                    const double bnorm = fabs(qtf), dq = delta / qnorm, sd = sgnorm / delta;
                    double tmp = (bnorm / gnorm) * (bnorm / qnorm) * sd;
                    tmp = tmp - dq * sd * sd + sqrt((tmp - dq) * (tmp - dq) + (1.0 - dq * dq) * (1.0 - sd * sd));
                    alpha = (dq * (1.0 - sd * sd)) / tmp;
                }
            }
            step = (1.0 - alpha) * fmin(sgnorm, delta) * w + alpha * xgn;
        }
        p = -step; xt = x + p; pnorm = fabs(d * p);
        if (iter == 1) delta = fmin(delta, pnorm);
        phase = 2;
    }
    // step(): one function evaluation + bookkeeping; returns true when finished (root estimate in x).
    // Single evaluation site and single dogleg site: lanes in different phases share both.
    SAT_DEV double next_x() const { return (phase == 0) ? x : ((phase == 1) ? x + h : xt); }
    SAT_DEV bool step() { return consume(f(next_x())); }
    // Warm start for a known initial guess: the first two evaluation points of hybrd (x0, then x0 + sqrt(eps)|x0| for the
    // forward-difference Jacobian) depend on the guess only, so the caller supplies sin/cos at those two points (computed
    // once per CTA with the same sincos) and the two trips through the shared evaluation site are saved. Same arithmetic.
    SAT_DEV void init_warm(const F& fn, double x0, const double sc[4]) {
        init(fn, x0);
        consume(f.at(sc[0], sc[1]));          // phase 0: f(x0)
        consume(f.at(sc[2], sc[3]));          // phase 1: f(x0 + h); never finishes, leaves the first trial point in xt
    }
    // bookkeeping for the value fe of f at next_x(); returns true when finished (root estimate in x)
    SAT_DEV bool consume(const double fe) {
        const double epsmch = 2.220446049250313e-16, xtol = 1.49012e-08, factor = 100.0;
        const int maxfev = 400;
        ++nfev;
        bool need_dogleg = false, finished = false;
        if (phase == 0) { fv = fe; fnorm = fabs(fv); start_outer(); }
        else if (phase == 1) {
            const double a = (fe - fv) / h;
            r = -a; q = (a != 0.0) ? -1.0 : 1.0;
            if (iter == 1) {
                d = (fabs(a) != 0.0) ? fabs(a) : 1.0;
                xnorm = fabs(d * x);
                delta = factor * xnorm;
                if (delta == 0.0) delta = factor;
            }
            qtf = q * fv;
            d = fmax(d, fabs(a));
            jeval = true;
            need_dogleg = true;
        } else {
            const double ft = fe;
            const double fnorm1 = fabs(ft);
            // zdiv: a zero numerator (exact root; exactly-zero predicted residual of the 1-D Newton step, i.e. nearly every
            // iteration) would take the whole warp through the division's zero/denormal slow path; 0 / b is +0 here
            const double qa = zdiv(fnorm1, fnorm);
            const double actred = (fnorm1 < fnorm) ? 1.0 - qa * qa : -1.0;
            const double pred = qtf + r * p;
            const double qp = zdiv(fabs(pred), fnorm);
            const double prered = (fabs(pred) < fnorm) ? 1.0 - qp * qp : 0.0;
            // prered == 1 exactly whenever the predicted residual is 0 (the usual full Newton step): x / 1 == x
            const double ratio = (prered > 0.0) ? ((prered == 1.0) ? actred : actred / prered) : 0.0;
            if (ratio < 0.1) { ncsuc = 0; ++ncfail; delta = 0.5 * delta; }
            else {
                ncfail = 0; ++ncsuc;
                if (ratio >= 0.5 || ncsuc > 1) delta = fmax(delta, pnorm * 2.0);      // pnorm / 0.5 (MINPACK: pnorm/p5), exact
                if (fabs(ratio - 1.0) <= 0.1) delta = pnorm * 2.0;
            }
            if (ratio >= 1e-4) { x = xt; fv = ft; xnorm = fabs(d * x); fnorm = fnorm1; ++iter; }
            ++nslow1; if (actred >= 1e-3) nslow1 = 0;
            if (jeval) ++nslow2;
            if (actred >= 0.1) nslow2 = 0;
            if (delta <= xtol * xnorm || fnorm == 0.0) finished = true;                     // info 1
            else if (nfev >= maxfev) finished = true;                                       // info 2
            else if (0.1 * fmax(0.1 * delta, pnorm) <= epsmch * xnorm) finished = true;     // info 3
            else if (nslow2 == 5 || nslow1 == 10) finished = true;                          // info 4 / 5
            else if (ncfail == 2) start_outer();                                            // re-evaluate the Jacobian
            else {
                // Broyden rank-1 update. pnorm is |d p| from the dogleg step with these same d and p, so (d p) / pnorm is
                // exactly +-1 for every finite non-zero d p: one IEEE division less per trial step, same bits
                const double dp = d * p;
                const double sgn = (dp != 0.0 && fabs(dp) <= 1.7976931348623157e308) ? copysign(1.0, dp) : dp / pnorm;
                const double s = q * ft, v = (s - pred) / pnorm, uu = d * sgn;
                if (ratio >= 1e-4) qtf = s;
                r = r + uu * v; jeval = false;
                need_dogleg = true;
            }
        }
        if (need_dogleg) dogleg();
        return finished;
    }
};

template <class F>
SAT_DEV double hybrd1(const F& fcn, double x0) {
    Hybrd1<F> s;
    s.init(fcn, x0);
    while (!s.step()) {}
    return s.x;
}

struct DzDebug { double rf_max, rf_min, r_ft, alpha0, alpha1, theta, dvm, f_cx; };

// ------------------------------------------------------------------------------------------
// Danger-zone count for one environment, evaluated by a LANE PAIR in three phases so that the expensive,
// data-dependent part (the fsolve iterations) can be compacted across the CTA:
//   dz_prepare  : each lane converts its own craft to orbital elements, the pair swaps them with shfl.xor 1,
//                 and each lane sets up ONE relative node (lane 0: node 1, lane 1: node 2): reachability test,
//                 theta, dVm and the two frozen-coefficient root problems (alpha_guess = +pi/2, -pi/2)
//   solve tasks : alpha = hybrd1(PFai{A, sth, dvm}, guess) -- independent work items; the kernels push them
//                 into a shared-memory queue and run them densely packed (only ~1/4 of the lanes have any)
//   dz_finalize : rf extremes from the two roots, interval test, pair sum -> 0/1/2
// environment.py:317-332 -> satellite_function.py:18-99, 317-373, 462-556. dz_prepare and dz_finalize contain
// warp-wide shuffles and MUST be called by all 32 lanes; `active` predicates the work.
// ------------------------------------------------------------------------------------------
struct DzNode {
    // state of one node's reachability problem between the phases
    double u, r_c, sq_e_sin, sq_k, dvm, sth, cth, r_ft;
    double A0, A1;          // P_fai coefficient for the +pi/2 and -pi/2 guesses (frozen at the guess, :518-523)
    int status;             // -1: element set for which the reference raises; 0: inactive; 1: unreachable (rf = 0,0); 2: two solves
    double theta, f_cx;     // diagnostics
};

template <bool EXACT = true>
SAT_DEV void dz_prepare(int craft, bool active, const double Ri[3], const double Vi[3], double fuel_c,
                        double u_grav, DzNode& nd) {
    nd.status = 0; nd.dvm = 0.0; nd.theta = 0.0; nd.f_cx = 0.0; nd.r_ft = 0.0;
    nd.A0 = 0.0; nd.A1 = 0.0; nd.sth = 0.0; nd.cth = 1.0; nd.sq_e_sin = 0.0; nd.sq_k = 0.0; nd.r_c = 0.0; nd.u = u_grav;
    if (!__any_sync(0xffffffffu, active)) return;          // warp-uniform: nothing to evaluate (all done / skipped)
    Elements el_own = {0, 0, 0, 0, 0, 0};
    int ok = 0;
    if (active) ok = orbital_elements<EXACT>(u_grav, Ri, Vi, el_own) ? 1 : 0;
    Elements el_oth;
    el_oth.a = __shfl_xor_sync(0xffffffffu, el_own.a, 1); el_oth.e = __shfl_xor_sync(0xffffffffu, el_own.e, 1);
    el_oth.i = __shfl_xor_sync(0xffffffffu, el_own.i, 1); el_oth.omega = __shfl_xor_sync(0xffffffffu, el_own.omega, 1);
    el_oth.Omega = __shfl_xor_sync(0xffffffffu, el_own.Omega, 1); el_oth.f = __shfl_xor_sync(0xffffffffu, el_own.f, 1);
    const int ok_both = ok & __shfl_xor_sync(0xffffffffu, ok, 1);
    const bool lane0 = craft == 0;
    const Elements& c = lane0 ? el_own : el_oth;     // pursuer
    const Elements& t = lane0 ? el_oth : el_own;     // target
    // Quantities both nodes of an env share are evaluated ONCE per lane pair: the two lanes put different arguments
    // through the same call and swap the results (every lane of the warp takes part in the shuffles; values of
    // inactive lanes are never used).
    // (1) sin/cos of the two inclinations: each lane its own craft's
    const double2 sci = Lm<EXACT>::sincos(el_own.i);
    const double si_x = __shfl_xor_sync(0xffffffffu, sci.x, 1), ci_x = __shfl_xor_sync(0xffffffffu, sci.y, 1);
    const double si_c = lane0 ? sci.x : si_x, ci_c = lane0 ? sci.y : ci_x;
    const double si_t = lane0 ? si_x : sci.x, ci_t = lane0 ? ci_x : sci.y;
    // (2) lane 0: sin/cos of the pursuer's true anomaly; lane 1: of Omega_c - Omega_t
    const double2 sc2 = Lm<EXACT>::sincos(lane0 ? c.f : c.Omega - t.Omega);
    const double s2_x = __shfl_xor_sync(0xffffffffu, sc2.x, 1), c2_x = __shfl_xor_sync(0xffffffffu, sc2.y, 1);
    const double sf0 = lane0 ? sc2.x : s2_x, cf0 = lane0 ? sc2.y : c2_x;
    const double sdo = lane0 ? s2_x : sc2.x, cdo = lane0 ? c2_x : sc2.y;
    // (3) calculate_latitudinal_angle, satellite_function.py:326-337: lane 0 -> temp1 / u_c1, lane 1 -> temp2 / u_t1.
    // sin/cos of (Omega_t - Omega_c) = -(Omega_c - Omega_t) follow from the exact odd/even symmetry of __sin / __cos.
    const double si_a = lane0 ? si_t : si_c, ci_a = lane0 ? ci_t : ci_c;
    const double si_b = lane0 ? si_c : si_t, ci_b = lane0 ? ci_c : ci_t;
    double temp = (si_a * (lane0 ? sdo : -sdo)) / (ci_a * si_b - si_a * ci_b * cdo);
    const double temp_x = __shfl_xor_sync(0xffffffffu, temp, 1);
    if (isnan(temp) || isnan(temp_x)) temp = 1.0;                        // :331-332 (both are replaced)
    const double u_own = Lm<EXACT>::atan(temp);
    const double u_x = __shfl_xor_sync(0xffffffffu, u_own, 1);
    const double u_c1 = lane0 ? u_own : u_x, u_t1 = lane0 ? u_x : u_own;
    // (4) squares (python `**`, i.e. libm pow): lane 0 -> e_c^2 and k^2, lane 1 -> e_t^2 and Delta_V_c^2
    const double e2_own = Lm<EXACT>::pow2(el_own.e);
    const double e2_x = __shfl_xor_sync(0xffffffffu, e2_own, 1);
    const double e2_c = lane0 ? e2_own : e2_x, e2_t = lane0 ? e2_x : e2_own;
    const double k = 1.0 + c.e * cf0;
    const double dv = fuel_c;                                             // Delta_V_c (:328)
    const double sq_own = Lm<EXACT>::pow2(lane0 ? k : dv);
    const double sq_x = __shfl_xor_sync(0xffffffffu, sq_own, 1);
    const double k2 = lane0 ? sq_own : sq_x, dv2 = lane0 ? sq_x : sq_own;
    // ---- no shuffles below this line
    if (!active) return;
    if (!ok_both) { nd.status = -1; return; }
    // :352-355; lane 0 -> node 1 (f_c1, r_ft1 uses f_t2), lane 1 -> node 2 (f_c2, r_ft2 uses f_t1) (Q5)
    const double f_cx = (lane0 ? u_c1 : kPi + u_c1) - c.omega;
    const double f_tx = (lane0 ? u_t1 + kPi : u_t1) - t.omega;
    nd.f_cx = f_cx;
    nd.r_ft = (t.a * (1.0 - e2_t)) / (1.0 + t.e * Lm<EXACT>::cos(f_tx));       // :363 / :365
    const double one_m_e2 = 1.0 - e2_c;
    const double r_c = c.a * one_m_e2 / k;                                // :57
    const double p_c = c.a * one_m_e2;                                    // :58
    // rf_extreme_point, satellite_function.py:462-494 with fai = 0
    const double df = f_cx - c.f;
    const double2 scdf = Lm<EXACT>::sincos(df);
    const double sdf = scdf.x, cdf = scdf.y;
    const double tmp1 = Lm<EXACT>::pow2(sdf) / (u_grav * k2 / (p_c * dv2) - 1.0);   // :466 / :481
    if (!(0.0 <= tmp1)) { nd.status = 1; return; }                                    // :478 -> (0, 0)
    // :469-470 with tan(fai) = 0: beta = atan(+-0 / sdf) = +-0 for every finite non-zero sdf, so cos(beta) = 1 and the
    // subtracted term u k^2 sin(beta)^2 / p_c is +-0 (u k^2 finite, p_c non-zero): dvm = sqrt(dv^2) bit for bit. The general
    // form stays for the other inputs; the shortcut keeps a zero-numerator division (warp-wide slow path), an atan and a
    // sincos off the common path.
    double cb, dvm;
    if (sdf != 0.0 && fabs(sdf) <= 1.0 && fabs(u_grav * k2) <= 1.7976931348623157e308 && p_c != 0.0 && p_c == p_c) {
        cb = 1.0;
        dvm = sqrt(dv2);
    } else {
        const double2 scb = Lm<EXACT>::sincos(Lm<EXACT>::atan(0.0 / sdf));       // :469
        cb = scb.y;
        dvm = sqrt(dv2 - u_grav * k2 * Lm<EXACT>::pow2(scb.x) / p_c);               // :470
    }
    // :464, :473-476 (theta stays 0 outside both ranges, Q5). One acos for the warp, the range decides how it is used:
    // an if / else-if around two acos calls made every warp run the routine twice with part of its lanes.
    const double ac = Lm<EXACT>::acos(cdf * 1.0);
    const bool in_a = (-kTwoPi <= df && df < -kPi) || (0.0 <= df && df < kPi);
    const bool in_b = (-kPi <= df && df < 0.0) || (kPi <= df && df < kTwoPi);
    const double theta = in_a ? ac : (in_b ? kTwoPi - ac : 0.0);
    const double2 scth = Lm<EXACT>::sincos(theta);
    const double sth = scth.x, cth = scth.y;
    const double sq = sqrt(u_grav / p_c);
    const double sq_e_sin = sq * c.e * sf0;                                           // :518 first term
    const double sq_k = sq * k * cb;                                                  // :519 first term
    nd.r_c = r_c; nd.sq_e_sin = sq_e_sin; nd.sq_k = sq_k; nd.dvm = dvm; nd.sth = sth; nd.cth = cth; nd.theta = theta;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        // alpha_guess = +-pi/2 (:516 / :534): libm gives sin(+-pi/2) = +-1 and cos(+-pi/2) = 6.123233995736766e-17 (the double
        // nearest pi/2 is below it); checked against glibm in tests/test_glibm_host.py
        const double sg = (j == 0) ? 1.0 : -1.0, cg = 6.123233995736766e-17;
        const double v1x = sq_e_sin + dvm * cg;
        const double v1y = sq_k + dvm * sg;
        const double h = r_c * v1y;                                                   // :521
        // :560. theta == 0 (45 % of the nodes the env visits) gives (+0) / (h v1y) - (+-0) / v1y = +-0 when the
        // denominators are non-zero numbers and v1x is finite; the sign of that zero is never observed (dz_degenerate),
        // and skipping the two zero-numerator divisions keeps the warp off the division slow path
        const double hv = h * v1y;
        double A;
        if (sth == 0.0 && cth == 1.0 && hv != 0.0 && hv == hv && v1y != 0.0 && fabs(v1x) <= 1.7976931348623157e308) A = 0.0;
        else A = (2.0 * u_grav * (1.0 - cth)) / hv - v1x * sth / v1y;
        if (j == 0) nd.A0 = A; else nd.A1 = A;
    }
    nd.status = 2;
}

// one root problem: satellite_function.py:523 / :540 -> :558-565
SAT_DEV double dz_guess(int j) { return (j == 0) ? kPi / 2 : -kPi / 2; }
// theta == 0 (Q5) makes P_fai identically zero: fsolve returns its initial guess unchanged after 3
// evaluations (|f| == 0 exit). Exact shortcut; 45 % of the solves on env-visited states.
SAT_DEV bool dz_degenerate(double A, double sth, double dvm) { return A == 0.0 && sth == 0.0 && fabs(dvm) <= 1.7976931348623157e308; }

template <bool EXACT = true>
SAT_DEV double dz_rf(const DzNode& nd, double alpha) {
    const double2 sc = Lm<EXACT>::sincos(alpha);
    const double s = sc.x, c = sc.y;
    const double v1x = nd.sq_e_sin + nd.dvm * c;                                      // :525 / :541
    const double v1y = nd.sq_k + nd.dvm * s;                                          // :526 / :542
    const double hm = nd.r_c * v1y;
    return fabs(Lm<EXACT>::pow2(hm) / (nd.u * (1.0 - nd.cth) + hm * v1y * nd.cth - hm * v1x * nd.sth));   // :530 / :545, :549-550
}

// returns 0/1/2, or -1 when the reference would raise; alpha0/alpha1 are ignored unless nd.status == 2
template <bool EXACT = true>
SAT_DEV int dz_finalize(bool active, const DzNode& nd, double alpha0, double alpha1, DzDebug* dbg) {
    int inside = 0;
    double rf_max = 0.0, rf_min = 0.0;
    if (nd.status == 2) {
        const double r0 = dz_rf<EXACT>(nd, alpha0), r1 = dz_rf<EXACT>(nd, alpha1);
        if (r0 < r1) { rf_max = r1; rf_min = r0; } else { rf_max = r0; rf_min = r1; }    // :551-554
    }
    if (nd.status >= 1) inside = (rf_min <= nd.r_ft && nd.r_ft <= rf_max) ? 1 : 0;        // :367-372
    if (dbg) {
        dbg->rf_max = rf_max; dbg->rf_min = rf_min; dbg->r_ft = nd.r_ft; dbg->f_cx = nd.f_cx;
        dbg->alpha0 = nd.status == 2 ? alpha0 : 0.0; dbg->alpha1 = nd.status == 2 ? alpha1 : 0.0;
        dbg->theta = nd.theta; dbg->dvm = nd.dvm;
    }
    const int inside_sum = inside + __shfl_xor_sync(0xffffffffu, inside, 1);
    const int bad = (nd.status < 0) ? 1 : 0;
    const int bad_any = bad | __shfl_xor_sync(0xffffffffu, bad, 1);
    if (!active) return 0;
    return bad_any ? -1 : inside_sum;
}

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), counter = (row_lo, row_hi, step_lo, step_hi), key = seed
// ------------------------------------------------------------------------------------------
SAT_DEV void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

}  // namespace sat
