/*
 * sat_oracle.c -- CPU restatement of the PPO-RL-Satellite hot path.
 * TEST INFRASTRUCTURE ONLY (see sat_oracle.h). Plain C, scalar, literal: it follows the
 * reference's expression order rather than any optimised form, so that it can be pinned
 * bit-for-bit against the reference where the arithmetic is IEEE-exact (+,-,*,/,sqrt,fma).
 *
 * Compile with -ffp-contract=off so the only fused operations are the explicit fma() calls
 * that reproduce OpenBLAS' ddot/dgemv kernels.
 */
#include "sat_oracle.h"
#include <math.h>
#include <float.h>
#include <string.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_PI 3.141592653589793
/* python/numpy scalar `x ** 2` is libm pow(x, 2.0), which is NOT always equal to x*x (glibc pow is
 * not correctly rounded: 90 of 1e5 random squares differ by one ulp). Keep the call: the Makefile passes
 * -fno-builtin-pow so that GCC does not fold it into x*x. */
#define SQ(x) pow((x), 2.0)
/* The RK4 script is evaluated on numpy ARRAYS in the batched configurations ((6, N) states): there `x ** 2` takes numpy's
 * fast path np.square = x*x (only exponents 2, 0.5, 1, 0, -1 have one; r ** 3 and r ** 5 stay libm pow). */
#define SQA(x) ((x) * (x))

/* ------------------------------------------------------------------------------------------
 * numpy / OpenBLAS summation orders (probed in the build container, numpy 2.3.5 +
 * scipy-openblas 0.3.30 Haswell kernels; see DESIGN.md "numpy arithmetic the env relies on"):
 *   np.dot(a3, b3)      = fma(a2,b2, fma(a1,b1, a0*b0))
 *   np.linalg.norm(a3)  = sqrt(np.dot(a3, a3))
 *   np.dot(M6x6, x6)[i] = ((p0+p2)+(p1+p3)) + fma(M[i][4],x4, M[i][5]*x5),  p_j = M[i][j]*x_j
 *   np.cross            = plain products and differences (no fusion)
 * ------------------------------------------------------------------------------------------ */
double orc_dot3(const double a[3], const double b[3]) {
    double s = a[0] * b[0];
    s = fma(a[1], b[1], s);
    s = fma(a[2], b[2], s);
    return s;
}
double orc_norm3(const double a[3]) { return sqrt(orc_dot3(a, a)); }

static void cross3(const double a[3], const double b[3], double c[3]) {
    double t0 = a[1] * b[2], t1 = a[2] * b[0], t2 = a[0] * b[1];
    double u0 = a[2] * b[1], u1 = a[0] * b[2], u2 = a[1] * b[0];
    c[0] = t0 - u0; c[1] = t1 - u1; c[2] = t2 - u2;
}

/* ------------------------------------------------------------------------------------------
 * RK4 script, 轨道外推-龙格库塔算法.py:15-30 (StateEq) and :34-40 (RungeKutta)
 * ------------------------------------------------------------------------------------------ */
void orc_state_eq(const double RV[6], double mu, double Re, double J2, double f[6]) {
    double x = RV[0], y = RV[1], z = RV[2];
    double r = sqrt(SQA(x) + SQA(y) + SQA(z));              /* :22 */
    double r3 = pow(r, 3.0), r5 = pow(r, 5.0);
    double gx = -mu * x / r3;                               /* :23-25 */
    double gy = -mu * y / r3;
    double gz = -mu * z / r3;
    double zr = z / r;
    double zr2 = SQA(zr);
    double c = -3.0 / 2.0 * J2 * SQA(Re) * mu;              /* python evaluates this scalar prefix left to right */
    double dgx = c * x / r5 * (1.0 - 5.0 * zr2);            /* :26-28 */
    double dgy = c * y / r5 * (1.0 - 5.0 * zr2);
    double dgz = c * z / r5 * (3.0 - 5.0 * zr2);
    f[0] = RV[3]; f[1] = RV[4]; f[2] = RV[5];
    f[3] = gx + dgx; f[4] = gy + dgy; f[5] = gz + dgz;      /* :29 */
}

void orc_rk4_step(double r0[6], double h, double mu, double Re, double J2) {
    double K1[6], K2[6], K3[6], K4[6], tmp[6];
    int i;
    orc_state_eq(r0, mu, Re, J2, K1);                       /* :35 */
    for (i = 0; i < 6; ++i) tmp[i] = r0[i] + h / 2.0 * K1[i];
    orc_state_eq(tmp, mu, Re, J2, K2);                      /* :36 */
    for (i = 0; i < 6; ++i) tmp[i] = r0[i] + h / 2.0 * K2[i];
    orc_state_eq(tmp, mu, Re, J2, K3);                      /* :37 */
    for (i = 0; i < 6; ++i) tmp[i] = r0[i] + h * K3[i];
    orc_state_eq(tmp, mu, Re, J2, K4);                      /* :38 */
    for (i = 0; i < 6; ++i)                                 /* :39 */
        r0[i] = r0[i] + h / 6.0 * (((K1[i] + 2.0 * K2[i]) + 2.0 * K3[i]) + K4[i]);
}

void orc_rk4_batch(double* x, int64_t n, int64_t ld, double h, int steps,
                   double mu, double re, double j2, int nthreads) {
    int64_t i;
#ifdef _OPENMP
    if (nthreads < 1) nthreads = 1;
#pragma omp parallel for num_threads(nthreads) schedule(static)
#endif
    for (i = 0; i < n; ++i) {
        double rv[6];
        int k, s;
        for (k = 0; k < 6; ++k) rv[k] = x[k * ld + i];
        for (s = 0; s < steps; ++s) orc_rk4_step(rv, h, mu, re, j2);
        for (k = 0; k < 6; ++k) x[k * ld + i] = rv[k];
    }
    (void)nthreads;
}

/* ------------------------------------------------------------------------------------------
 * Clohessy_Wiltshire.State_transition_matrix, satellite_function.py:753-781
 * ------------------------------------------------------------------------------------------ */
void orc_cw_matrix(double t, double M[36]) {
    double u = 3.986e14;                                    /* :750 */
    double R = 42164000.0;                                  /* :756 */
    double r = R;
    double omega = sqrt(u / (r * r * r));                   /* :761 (python int r**3 is exact: 7.4958e22 < 2^77 but not < 2^53: see note) */
    double tau, s, c;
    /* note: r ** 3 on the python int 42164000 is the exact integer 74958094340944000000000, and
     * u / int converts it to the nearest double; r*r*r in double is exact up to the same rounding
     * because 42164000^2 = 1.7778e15 < 2^53 and the last product rounds once. */
    tau = omega * t;                                        /* :763 */
    s = sin(tau); c = cos(tau);                             /* :764-765 */
    memset(M, 0, 36 * sizeof(double));
    M[0] = 4 - 3 * c;            M[3] = s / omega;            M[4] = 2 * (1 - c) / omega;      /* :767 */
    M[6] = 6 * (s - tau);        M[7] = 1; M[9] = -2 * (1 - c) / omega; M[10] = 4 * s / omega - 3 * tau; /* :768 */
    M[14] = c;                   M[17] = s / omega;                                            /* :769 */
    M[18] = 3 * omega * s;       M[21] = c;                  M[22] = 2 * s;                   /* :770 */
    M[24] = 6 * omega * (c - 1); M[27] = -2 * s;             M[28] = 4 * c - 3;               /* :771 */
    M[32] = -omega * s;          M[35] = c;                                                   /* :772 */
}

void orc_cw_apply(const double M[36], const double x[6], double out[6]) {   /* :778-779 np.dot */
    int i;
    for (i = 0; i < 6; ++i) {
        const double* r = M + 6 * i;
        double p0 = r[0] * x[0], p1 = r[1] * x[1], p2 = r[2] * x[2], p3 = r[3] * x[3];
        double head = (p0 + p2) + (p1 + p3);
        double tail = fma(r[4], x[4], r[5] * x[5]);
        out[i] = head + tail;
    }
}

/* ------------------------------------------------------------------------------------------
 * calculate_orbital_elements, satellite_function.py:161-255
 * ------------------------------------------------------------------------------------------ */
int orc_orbital_elements(double miu, const double R0[3], const double V0[3], double data[6]) {
    double r_norm = orc_norm3(R0);                          /* :183 */
    double v_norm = orc_norm3(V0);                          /* :184 */
    double r_dot_v = orc_dot3(R0, V0);                      /* :185 */
    double energy = 2 / r_norm - SQ(v_norm) / miu;          /* :186 */
    double a = 0, e, h, p, n, inc, omega = 0, Omega, f = 0, uu = 0;
    double E[3], H[3], N[3];
    double c1, c2;
    int k;
    if (energy != 0) a = 1 / fabs(energy);                  /* :188 */
    c1 = SQ(v_norm) / miu - 1 / r_norm;                     /* :193 */
    c2 = r_dot_v / miu;
    for (k = 0; k < 3; ++k) E[k] = c1 * R0[k] - c2 * V0[k];
    e = orc_norm3(E);                                       /* :194 */
    cross3(R0, V0, H);                                      /* :197 */
    h = orc_norm3(H);                                       /* :199 */
    p = SQ(h) / miu;                                        /* :201 */
    {   /* N = cross(Z, H), Z = [0,0,1]  :206 */
        double Z[3] = {0, 0, 1};
        cross3(Z, H, N);
    }
    n = orc_norm3(N);                                       /* :208 */
    inc = acos(H[2] / h);                                   /* :210  np.dot(Z,H) == H[2] */
    if (e != 0) {
        if (n != 0) omega = acos(orc_dot3(N, E) / n / e);   /* :214-217 */
        else omega = 0.0;
        if (E[2] < 0) omega = 2 * ORC_PI - omega;           /* :221 */
    } else {
        uu = acos(orc_dot3(N, R0) / n / r_norm);            /* :225 */
        if (R0[2] < 0) uu = 2 * ORC_PI - uu;
    }
    if (n != 0) Omega = acos(N[0] / n);                     /* :230-233 */
    else Omega = 0.0;
    if (N[1] < 0) Omega = 2 * ORC_PI - Omega;               /* :237 */
    if (e != 0) {
        f = acos(orc_dot3(E, R0) / e / r_norm);             /* :242 */
        if (r_dot_v < 0) f = 2 * ORC_PI - f;
    }
    if (energy != 0) {                                      /* :247-253 */
        if (e != 0) { data[0] = a; data[1] = e; data[2] = inc; data[3] = omega; data[4] = Omega; data[5] = f; return 6; }
        data[0] = a; data[1] = inc; data[2] = uu; data[3] = Omega; return 4;
    }
    data[0] = p; data[1] = inc; data[2] = omega; data[3] = Omega; data[4] = f; return 5;
}

/* calculate_state_information (6-element form), satellite_function.py:257-315 */
void orc_state_information(const double d[6], double miu, double R[3], double V[3]) {
    double a = d[0], e = d[1], i = d[2], omega = d[3], Omega = d[4], f = d[5];
    double p = fabs(a * (1 - SQ(e)));                       /* :285 */
    double u = omega + f;                                   /* :286 */
    double k = p / (1 + e * cos(f));                        /* :303 */
    double s;
    R[0] = k * (cos(Omega) * cos(u) - sin(Omega) * sin(u) * cos(i));
    R[1] = k * (sin(Omega) * cos(u) + cos(Omega) * sin(u) * cos(i));
    R[2] = k * (sin(i) * sin(u));
    s = pow(miu / p, 0.5);                                  /* :309 */
    V[0] = s * (-cos(Omega) * (sin(u) + e * sin(omega)) - sin(Omega) * (cos(u) + e * cos(omega)) * cos(i));
    V[1] = s * (-sin(Omega) * (sin(u) + e * sin(omega)) + cos(Omega) * (cos(u) + e * cos(omega)) * cos(i));
    V[2] = s * (sin(i) * (cos(u) + e * cos(omega)));
}

/* ------------------------------------------------------------------------------------------
 * scipy.optimize.fsolve(func, x0) for n = 1: MINPACK hybrd with scipy defaults
 * (xtol=1.49012e-08, maxfev=400, factor=100, epsfcn->machine eps, mode 1). SURVEY.md Appendix B.
 * ------------------------------------------------------------------------------------------ */
double orc_fsolve1(orc_fn1 fcn, void* ctx, double x0, int* nfev_out, int* info_out) {
    const double epsmch = DBL_EPSILON, xtol = 1.49012e-08, factor = 100.0;
    const int maxfev = 400;
    const double p1 = 0.1, p5 = 0.5, p001 = 1e-3, p0001 = 1e-4;
    double x = x0, fv, fnorm, d = 0, delta = 0, xnorm = 0;
    int nfev, iter = 1, ncsuc = 0, ncfail = 0, nslow1 = 0, nslow2 = 0, info = 0;
    fv = fcn(x, ctx); nfev = 1;
    fnorm = fabs(fv);
    for (;;) {                                              /* outer: Jacobian refresh */
        int jeval = 1;
        double h = sqrt(epsmch) * fabs(x), a, r, q, qtf;
        if (h == 0) h = sqrt(epsmch);
        a = (fcn(x + h, ctx) - fv) / h; nfev++;
        r = -a; q = (a != 0) ? -1.0 : 1.0;
        if (iter == 1) {
            d = (fabs(a) != 0) ? fabs(a) : 1.0;
            xnorm = fabs(d * x);
            delta = factor * xnorm;
            if (delta == 0) delta = factor;
        }
        qtf = q * fv;
        d = fmax(d, fabs(a));
        for (;;) {                                          /* inner */
            double t, xgn, qnorm, step, p, xt, pnorm, ft, fnorm1, actred, pred, prered, ratio;
            /* dogleg */
            t = r; if (t == 0) { t = epsmch * fabs(r); if (t == 0) t = epsmch; }
            xgn = qtf / t; qnorm = fabs(d * xgn);
            if (qnorm <= delta) step = xgn;
            else {
                double w = (r * qtf) / d, gnorm = fabs(w), sgnorm = 0, alpha = delta / qnorm;
                if (gnorm != 0) {
                    double tt;
                    w = (w / gnorm) / d; tt = fabs(r * w); sgnorm = (gnorm / tt) / tt; alpha = 0;
                    if (sgnorm < delta) {
                        double bnorm = fabs(qtf);
                        double dq = delta / qnorm, sd = sgnorm / delta;
                        double tmp = (bnorm / gnorm) * (bnorm / qnorm) * sd;
                        tmp = tmp - dq * sd * sd + sqrt((tmp - dq) * (tmp - dq) + (1 - dq * dq) * (1 - sd * sd));
                        alpha = (dq * (1 - sd * sd)) / tmp;
                    }
                }
                step = (1 - alpha) * fmin(sgnorm, delta) * w + alpha * xgn;
            }
            p = -step; xt = x + p; pnorm = fabs(d * p);
            if (iter == 1) delta = fmin(delta, pnorm);
            ft = fcn(xt, ctx); nfev++;
            fnorm1 = fabs(ft);
            actred = (fnorm1 < fnorm) ? 1 - (fnorm1 / fnorm) * (fnorm1 / fnorm) : -1.0;
            pred = qtf + r * p;
            prered = (fabs(pred) < fnorm) ? 1 - (fabs(pred) / fnorm) * (fabs(pred) / fnorm) : 0.0;
            ratio = (prered > 0) ? actred / prered : 0.0;
            if (ratio < p1) { ncsuc = 0; ncfail++; delta = p5 * delta; }
            else {
                ncfail = 0; ncsuc++;
                if (ratio >= p5 || ncsuc > 1) delta = fmax(delta, pnorm / p5);
                if (fabs(ratio - 1) <= p1) delta = pnorm / p5;
            }
            if (ratio >= p0001) { x = xt; fv = ft; xnorm = fabs(d * x); fnorm = fnorm1; iter++; }
            nslow1++; if (actred >= p001) nslow1 = 0;
            if (jeval) nslow2++;
            if (actred >= p1) nslow2 = 0;
            if (delta <= xtol * xnorm || fnorm == 0) { info = 1; goto done; }
            if (nfev >= maxfev) { info = 2; goto done; }
            if (p1 * fmax(p1 * delta, pnorm) <= epsmch * xnorm) { info = 3; goto done; }
            if (nslow2 == 5) { info = 4; goto done; }
            if (nslow1 == 10) { info = 5; goto done; }
            if (ncfail == 2) break;
            {   /* Broyden rank-1 update */
                double s = q * ft, v = (s - pred) / pnorm, uu = d * ((d * p) / pnorm);
                if (ratio >= p0001) qtf = s;
                r = r + uu * v; jeval = 0;
            }
        }
    }
done:
    if (nfev_out) *nfev_out = nfev;
    if (info_out) *info_out = info;
    return x;
}

typedef struct { double A, sth, dvm; } pfai_ctx;
static double pfai_eq(double alpha, void* vctx) {           /* satellite_function.py:559-562 */
    pfai_ctx* c = (pfai_ctx*)vctx;
    return c->A * (c->dvm * cos(alpha)) + c->sth * (-c->dvm * sin(alpha));
}
double orc_numerical_iteration(double u, double Delta_Vm, double theta, double v_1x, double v_1y,
                               double h, double alpha_guess) {
    pfai_ctx c;
    c.A = (2 * u * (1 - cos(theta))) / (h * v_1y) - v_1x * sin(theta) / v_1y;
    c.sth = sin(theta);
    c.dvm = Delta_Vm;
    return orc_fsolve1(pfai_eq, &c, alpha_guess, 0, 0);     /* :564-565 */
}

/* ------------------------------------------------------------------------------------------
 * Time_window_of_danger_zone (the subset the env uses), satellite_function.py:18-99, 317-373, 462-565
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    double u, Delta_V_c;
    double a_c, e_c, i_c, omega_c, Omega_c, f0_c, r_c, p_c;
    double a_t, e_t, i_t, omega_t, Omega_t, f0_t;
} tw_ctx;

static void rf_extreme_point(const tw_ctx* s, double f_cx, double* rf_max_out, double* rf_min_out, double* dbg) {
    const double fai = 0.0;                                 /* :33 */
    double Delta_Vm = 0, beta = 0, theta = 0;               /* :464 */
    double df = f_cx - s->f0_c;
    double sdf = sin(df);
    double k = (1 + s->e_c * cos(s->f0_c));
    double temp1 = SQ(sdf) / (s->u * SQ(k) / (s->p_c * SQ(s->Delta_V_c)) - 1);   /* :466 / :481 */
    double sq, v_1x, v_1y, h, alpha, rf_max, rf_min, v_1x_m, v_1y_m, h_m, sb;
    if (0 <= temp1) {
        beta = atan(tan(fai) / sdf);                        /* :469 */
        sb = sin(beta);
        Delta_Vm = sqrt(SQ(s->Delta_V_c) - s->u * SQ(k) * SQ(sb) / s->p_c);  /* :470 */
        if ((-2 * ORC_PI <= df && df < -ORC_PI) || (0 <= df && df < ORC_PI))                /* :473 */
            theta = acos(cos(df) * cos(fai));
        else if ((-ORC_PI <= df && df < 0) || (ORC_PI <= df && df < 2 * ORC_PI))            /* :475 */
            theta = 2 * ORC_PI - acos(cos(df) * cos(fai));
    } else { *rf_max_out = 0; *rf_min_out = 0; if (dbg) { dbg[3] = dbg[4] = dbg[5] = dbg[6] = 0; } return; }    /* :478 */

    sq = sqrt(s->u / s->p_c);
    /* first extreme, alpha_guess = +pi/2  :516-531 */
    {
        double ag = ORC_PI / 2;
        v_1x = sq * s->e_c * sin(s->f0_c) + Delta_Vm * cos(ag);
        v_1y = sq * (1 + s->e_c * cos(s->f0_c)) * cos(beta) + Delta_Vm * sin(ag);
        h = s->r_c * v_1y;
        alpha = orc_numerical_iteration(s->u, Delta_Vm, theta, v_1x, v_1y, h, ag);
        v_1x_m = sq * s->e_c * sin(s->f0_c) + Delta_Vm * cos(alpha);
        v_1y_m = sq * (1 + s->e_c * cos(s->f0_c)) * cos(beta) + Delta_Vm * sin(alpha);
        h_m = s->r_c * v_1y_m;
        rf_max = SQ(h_m) / (s->u * (1 - cos(theta)) + h_m * v_1y_m * cos(theta) - h_m * v_1x_m * sin(theta));
        if (dbg) dbg[3] = alpha;
    }
    /* second extreme, alpha_guess = -pi/2  :534-547 */
    {
        double ag = -ORC_PI / 2;
        v_1x = sq * s->e_c * sin(s->f0_c) + Delta_Vm * cos(ag);
        v_1y = sq * (1 + s->e_c * cos(s->f0_c)) * cos(beta) + Delta_Vm * sin(ag);
        h = s->r_c * v_1y;
        alpha = orc_numerical_iteration(s->u, Delta_Vm, theta, v_1x, v_1y, h, ag);
        v_1x_m = sq * s->e_c * sin(s->f0_c) + Delta_Vm * cos(alpha);
        v_1y_m = sq * (1 + s->e_c * cos(s->f0_c)) * cos(beta) + Delta_Vm * sin(alpha);
        h_m = s->r_c * v_1y_m;
        rf_min = SQ(h_m) / (s->u * (1 - cos(theta)) + h_m * v_1y_m * cos(theta) - h_m * v_1x_m * sin(theta));
        if (dbg) { dbg[4] = alpha; dbg[5] = theta; dbg[6] = Delta_Vm; }
    }
    rf_max = fabs(rf_max); rf_min = fabs(rf_min);           /* :549-554 */
    if (rf_max < rf_min) { double t = rf_min; rf_min = rf_max; rf_max = t; }
    *rf_max_out = rf_max; *rf_min_out = rf_min;
}

int orc_danger_zone(const double R0_c[3], const double V0_c[3], const double R0_t[3], const double V0_t[3],
                    double Delta_V_c, double u) {
    return orc_danger_zone_debug(R0_c, V0_c, R0_t, V0_t, Delta_V_c, u, 0);
}

/* dbg (nullable) [2][8]: per node rf_max, rf_min, r_ft, alpha(+pi/2), alpha(-pi/2), theta, dVm, f_c */
int orc_danger_zone_debug(const double R0_c[3], const double V0_c[3], const double R0_t[3], const double V0_t[3],
                          double Delta_V_c, double u, double* dbg) {
    tw_ctx s;
    double el[6];
    double temp1, temp2, u_c1, u_c2, u_t1, u_t2, f_c1, f_c2, f_t1, f_t2;
    double rf_max_c1, rf_min_c1, rf_max_c2, rf_min_c2, r_ft1, r_ft2;
    int in1, in2;
    s.u = u; s.Delta_V_c = Delta_V_c;
    if (orc_orbital_elements(u, R0_c, V0_c, el) != 6) return -1;                 /* :52-58 */
    s.a_c = el[0]; s.e_c = el[1]; s.i_c = el[2]; s.omega_c = el[3]; s.Omega_c = el[4]; s.f0_c = el[5];
    s.r_c = s.a_c * (1 - SQ(s.e_c)) / (1 + s.e_c * cos(s.f0_c));
    s.p_c = s.a_c * (1 - SQ(s.e_c));
    if (orc_orbital_elements(u, R0_t, V0_t, el) != 6) return -1;                 /* :81-86 */
    s.a_t = el[0]; s.e_t = el[1]; s.i_t = el[2]; s.omega_t = el[3]; s.Omega_t = el[4]; s.f0_t = el[5];

    /* calculate_latitudinal_angle :317-339 */
    temp1 = (sin(s.i_t) * sin(s.Omega_c - s.Omega_t)) /
            (cos(s.i_t) * sin(s.i_c) - sin(s.i_t) * cos(s.i_c) * cos(s.Omega_c - s.Omega_t));
    temp2 = (sin(s.i_c) * sin(s.Omega_t - s.Omega_c)) /
            (cos(s.i_c) * sin(s.i_t) - sin(s.i_c) * cos(s.i_t) * cos(s.Omega_t - s.Omega_c));
    if (isnan(temp1) || isnan(temp2)) { temp1 = 1; temp2 = 1; }
    u_c1 = atan(temp1); u_c2 = ORC_PI + u_c1;
    u_t1 = atan(temp2); u_t2 = u_t1 + ORC_PI;
    /* calculate_number_of_hanger_area :341-373 */
    f_c1 = u_c1 - s.omega_c; f_c2 = u_c2 - s.omega_c;
    f_t1 = u_t1 - s.omega_t; f_t2 = u_t2 - s.omega_t;
    rf_extreme_point(&s, f_c1, &rf_max_c1, &rf_min_c1, dbg);
    rf_extreme_point(&s, f_c2, &rf_max_c2, &rf_min_c2, dbg ? dbg + 8 : 0);
    r_ft1 = (s.a_t * (1 - SQ(s.e_t))) / (1 + s.e_t * cos(f_t2));            /* :363 (swapped, Q5) */
    r_ft2 = (s.a_t * (1 - SQ(s.e_t))) / (1 + s.e_t * cos(f_t1));            /* :365 */
    if (dbg) {
        dbg[0] = rf_max_c1; dbg[1] = rf_min_c1; dbg[2] = r_ft1; dbg[7] = f_c1;
        dbg[8] = rf_max_c2; dbg[9] = rf_min_c2; dbg[10] = r_ft2; dbg[15] = f_c2;
    }
    in1 = (rf_min_c1 <= r_ft1 && r_ft1 <= rf_max_c1);
    in2 = (rf_min_c2 <= r_ft2 && r_ft2 <= rf_max_c2);
    if (in1 && in2) return 2;
    if (in1 || in2) return 1;
    return 0;
}

/* ------------------------------------------------------------------------------------------
 * environment.satellites, environment.py:26-179 (Flag 0) / :181-255 (Flag 1)
 * ------------------------------------------------------------------------------------------ */
static double g_terms[7];
void orc_env_last_terms(double out[7]) { memcpy(out, g_terms, sizeof(g_terms)); }

void orc_env_init(orc_env* e, double d_capture, double d_range, double fuel_c, double fuel_t,
                  int max_episode_steps) {
    memset(e, 0, sizeof(*e));
    e->d_capture = d_capture; e->d_range = d_range;         /* :35,45 */
    e->fuel_c = fuel_c; e->fuel_t = fuel_t;                 /* :42-43 */
    e->dis = INFINITY;                                      /* :44 */
    e->dangerous_zone = 0;                                  /* :41 */
    e->max_episode_steps = max_episode_steps;               /* :46 */
}

static void make_obs(const orc_env* e, double obs[18]) {    /* :76-77 layout */
    int k;
    for (k = 0; k < 3; ++k) {
        obs[k] = e->P[k] - e->E[k];
        obs[3 + k] = e->Pv[k] - e->Ev[k];
        obs[6 + k] = e->P[k]; obs[9 + k] = e->Pv[k];
        obs[12 + k] = e->E[k]; obs[15 + k] = e->Ev[k];
    }
}

void orc_env_reset(orc_env* e, int flag, double obs[18]) {  /* :66-79; fuel/dis/dangerous_zone persist (Q2) */
    e->P[0] = 200000; e->P[1] = 0; e->P[2] = 0;
    e->Pv[0] = e->Pv[1] = e->Pv[2] = 0;
    e->E[0] = 18000; e->E[1] = 0; e->E[2] = 0;
    e->Ev[0] = e->Ev[1] = e->Ev[2] = 0;
    e->flag = flag;
    e->int_state = 1;
    if (obs) make_obs(e, obs);
}

static double clip16(double a) { return a < -1.6 ? -1.6 : (a > 1.6 ? 1.6 : a); }   /* np.clip :86 */

/* impulse application incl. the int64 truncation quirk Q1 (:93-104) */
static void add_dv(orc_env* e, double v[3], const double a[3]) {
    int k;
    for (k = 0; k < 3; ++k) {
        double s = v[k] + a[k];
        v[k] = e->int_state ? trunc(s) : s;
    }
}

static double cosine3(const double a[3], const double b[3]) {       /* :351-353 pattern */
    double na = orc_norm3(a), nb = orc_norm3(b), ua[3], ub[3];
    int k;
    for (k = 0; k < 3; ++k) { ua[k] = a[k] / na; ub[k] = b[k] / nb; }
    return orc_dot3(ua, ub);
}

/* shared front half of step(): clip, gate, impulse, fuel. returns previous distance */
static double step_impulse(orc_env* e, const double pa_in[3], const double ea_in[3], double pa[3], double ea[3]) {
    double d[3], dis_prev;
    int k;
    for (k = 0; k < 3; ++k) { pa[k] = clip16(pa_in[k]); ea[k] = clip16(ea_in[k]); }      /* :86-87 */
    for (k = 0; k < 3; ++k) d[k] = e->P[k] - e->E[k];
    dis_prev = orc_norm3(d);                                                             /* :89 */
    if (e->flag == 0 || e->flag == 2) {                                                  /* Flag 2: :265-277, same gating */
        if (e->dis < e->d_range && e->dangerous_zone != 0) {                             /* :91-96 */
            add_dv(e, e->Ev, ea);
            if (e->int_state) { for (k = 0; k < 3; ++k) e->Pv[k] = trunc(e->Pv[k] + 0); }
            pa[0] = pa[1] = pa[2] = 0;
        } else { add_dv(e, e->Pv, pa); add_dv(e, e->Ev, ea); }                           /* :97-104 */
    } else {
        if (e->dangerous_zone != 0) { add_dv(e, e->Pv, pa); add_dv(e, e->Ev, ea); }      /* :190-193 */
        else { add_dv(e, e->Pv, pa); ea[0] = ea[1] = ea[2] = 0; }                        /* :194-198 */
    }
    e->fuel_c -= (fabs(pa[0]) + fabs(pa[1])) + fabs(pa[2]);                              /* :106 */
    e->fuel_t -= (fabs(ea[0]) + fabs(ea[1])) + fabs(ea[2]);                              /* :107 */
    return dis_prev;
}

/* shared back half of step(): distance, terminal checks, danger zone, reward */
static int step_finish(orc_env* e, double dis_prev, const double pa[3], int episode_count,
                       double obs[18], double* reward) {
    double d[3], a, b, c, pv1, pv2, pv3, pv4, r;
    int k;
    e->int_state = 0;
    for (k = 0; k < 3; ++k) d[k] = e->P[k] - e->E[k];
    e->dis = orc_norm3(d);                                                               /* :132 */
    make_obs(e, obs);
    if (e->flag == 2) {                                  /* :303-316: reward 0, danger zone not re-evaluated; the surrogate
                                                            fit between (:295-301) is outside the hot path */
        *reward = 0.0;
        return (e->dis <= e->d_capture || episode_count >= e->max_episode_steps) ? 1 : 0;
    }
    if (e->dis <= e->d_capture) { *reward = (e->flag == 0) ? 100.0 : -150.0; return 1; } /* :139-142 / :221-225 */
    if (episode_count >= e->max_episode_steps) { *reward = (e->flag == 0) ? 0.0 : 100.0; return 1; } /* :144-147 / :227-231 */
    {   /* calculate_number_hanger_area :317-332, relative_state_to_absolute_state :334-343 */
        const double R_cw[3] = {27098000, 32306000, 0}, V_cw[3] = {-2350, 1970, 0};
        double Rc[3], Vc[3], Rt[3], Vt[3];
        int dz;
        for (k = 0; k < 3; ++k) {
            Rc[k] = R_cw[k] + e->P[k]; Vc[k] = V_cw[k] + e->Pv[k];
            Rt[k] = R_cw[k] + e->E[k]; Vt[k] = V_cw[k] + e->Ev[k];
        }
        dz = orc_danger_zone(Rc, Vc, Rt, Vt, e->fuel_c, 3.986e14);
        if (dz < 0) { e->err = 1; dz = 0; }
        e->dangerous_zone = dz;
    }
    a = (e->dis < dis_prev) ? 1 : -1;                                                    /* :161 */
    b = (e->d_capture <= e->dis && e->dis <= 4 * e->d_capture) ? -1 : -2;                /* :162 */
    c = (e->dangerous_zone == 0) ? -1 : e->dangerous_zone * 0.5;                         /* :164 */
    pv1 = cosine3(e->P, e->E);                                                           /* :166 -> :370-379 */
    pv2 = cosine3(e->Pv, e->Ev);                                                         /* :167 -> :346-354 */
    pv3 = cosine3(d, e->Pv);                                                             /* :168 -> :357-368 */
    if (pa[0] != 0 && pa[1] != 0 && pa[2] != 0) pv4 = -cosine3(d, pa);                   /* :169 -> :382-396 */
    else pv4 = 0;
    r = (a + b) + c;
    r = r + 1 * pv1;                                                                     /* :172-175 */
    r = r + 0.6 * pv2;
    r = r + 0.2 * pv3;
    r = r + 2 * pv4;
    g_terms[0] = a; g_terms[1] = b; g_terms[2] = c; g_terms[3] = pv1; g_terms[4] = pv2; g_terms[5] = pv3; g_terms[6] = pv4;
    *reward = (e->flag == 0) ? r : -r;                                                   /* :251 */
    return 0;
}

int orc_env_step(orc_env* e, const double M[36], const double pa_in[3], const double ea_in[3],
                 int episode_count, double obs[18], double* reward) {
    double pa[3], ea[3], sc[6], st[6], nc[6], nt[6], dis_prev;
    int k;
    dis_prev = step_impulse(e, pa_in, ea_in, pa, ea);
    for (k = 0; k < 3; ++k) { sc[k] = e->P[k]; sc[3 + k] = e->Pv[k]; st[k] = e->E[k]; st[3 + k] = e->Ev[k]; }
    orc_cw_apply(M, sc, nc);                                                             /* :117-121 */
    orc_cw_apply(M, st, nt);
    for (k = 0; k < 3; ++k) { e->P[k] = nc[k]; e->Pv[k] = nc[3 + k]; e->E[k] = nt[k]; e->Ev[k] = nt[3 + k]; }  /* :130-131 */
    return step_finish(e, dis_prev, pa, episode_count, obs, reward);
}

int orc_env_step_rk4(orc_env* e, double h, int substeps, double mu, double re, double j2,
                     const double pa_in[3], const double ea_in[3], int episode_count,
                     double obs[18], double* reward) {
    /* rk4 mode (SURVEY H8): same step with the CW matvec replaced by S RK4 substeps of the
     * inertial two-body(+J2) ODE; relative<->inertial is the reference's bare translation
     * (environment.py:334-343). */
    const double R_cw[3] = {27098000, 32306000, 0}, V_cw[3] = {-2350, 1970, 0};
    double pa[3], ea[3], sc[6], st[6], dis_prev;
    int k, s;
    dis_prev = step_impulse(e, pa_in, ea_in, pa, ea);
    for (k = 0; k < 3; ++k) {
        sc[k] = R_cw[k] + e->P[k]; sc[3 + k] = V_cw[k] + e->Pv[k];
        st[k] = R_cw[k] + e->E[k]; st[3 + k] = V_cw[k] + e->Ev[k];
    }
    for (s = 0; s < substeps; ++s) { orc_rk4_step(sc, h, mu, re, j2); orc_rk4_step(st, h, mu, re, j2); }
    for (k = 0; k < 3; ++k) {
        e->P[k] = sc[k] - R_cw[k]; e->Pv[k] = sc[3 + k] - V_cw[k];
        e->E[k] = st[k] - R_cw[k]; e->Ev[k] = st[3 + k] - V_cw[k];
    }
    return step_finish(e, dis_prev, pa, episode_count, obs, reward);
}

void orc_env_step_batch(orc_env* envs, int32_t* counts, int64_t n, const double M[36],
                        const double* pa, const double* ea, double* obs, double* reward,
                        uint8_t* done, int auto_reset, int nthreads) {
    int64_t i;
#ifdef _OPENMP
    if (nthreads < 1) nthreads = 1;
#pragma omp parallel for num_threads(nthreads) schedule(static)
#endif
    for (i = 0; i < n; ++i) {
        int d;
        counts[i] += 1;
        d = orc_env_step(&envs[i], M, pa + 3 * i, ea + 3 * i, counts[i], obs + 18 * i, &reward[i]);
        done[i] = (uint8_t)d;
        if (d && auto_reset) { orc_env_reset(&envs[i], envs[i].flag, obs + 18 * i); counts[i] = 0; }
    }
    (void)nthreads;
}

void orc_env_step_rk4_batch(orc_env* envs, int32_t* counts, int64_t n, double h, int substeps,
                            double mu, double re, double j2, const double* pa, const double* ea,
                            double* obs, double* reward, uint8_t* done, int auto_reset, int nthreads) {
    int64_t i;
#ifdef _OPENMP
    if (nthreads < 1) nthreads = 1;
#pragma omp parallel for num_threads(nthreads) schedule(static)
#endif
    for (i = 0; i < n; ++i) {
        int d;
        counts[i] += 1;
        d = orc_env_step_rk4(&envs[i], h, substeps, mu, re, j2, pa + 3 * i, ea + 3 * i, counts[i],
                             obs + 18 * i, &reward[i]);
        done[i] = (uint8_t)d;
        if (d && auto_reset) { orc_env_reset(&envs[i], envs[i].flag, obs + 18 * i); counts[i] = 0; }
    }
    (void)nthreads;
}

/* ------------------------------------------------------------------------------------------
 * normalization.py:7-63
 * ------------------------------------------------------------------------------------------ */
void orc_rms_update(orc_rms* r, const double* x) {          /* :19-29 */
    int k;
    r->n += 1;
    if (r->n == 1) {
        for (k = 0; k < r->dim; ++k) { r->mean[k] = x[k]; r->std[k] = x[k]; }           /* Q7 */
    } else {
        for (k = 0; k < r->dim; ++k) {
            double old_mean = r->mean[k];
            r->mean[k] = old_mean + (x[k] - old_mean) / (double)r->n;
            r->S[k] = r->S[k] + (x[k] - old_mean) * (x[k] - r->mean[k]);
            r->std[k] = sqrt(r->S[k] / (double)r->n);
        }
    }
}
void orc_normalize(orc_rms* r, const double* x, int update, double* out) {   /* :37-43 */
    int k;
    if (update) orc_rms_update(r, x);
    for (k = 0; k < r->dim; ++k) out[k] = (x[k] - r->mean[k]) / (r->std[k] + 1e-8);
}
double orc_reward_scaling(orc_rms* r, double* R, double gamma, double x) {   /* :56-60 */
    *R = gamma * (*R) + x;
    orc_rms_update(r, R);
    return x / (r->std[0] + 1e-8);
}

/* ------------------------------------------------------------------------------------------
 * GAE, ppo_continuous.py:198-210. Under numpy 2 (NEP 50) the recursion runs in float32:
 * delta and d are np.float32, gamma*lamda is a python float (weak) -> float32 arithmetic.
 * gamma and lamda are the python floats: their product is formed in double and rounded once.
 * ------------------------------------------------------------------------------------------ */
void orc_gae(const float* r, const float* vs, const float* vs_next, const float* dw, const float* done,
             int64_t B, double gamma, double lamda, float* adv, float* v_target) {
    int64_t t;
    float gae = 0.0f;
    const float gl = (float)(gamma * lamda);                 /* python float product, then weak-cast */
    const float g32 = (float)gamma;                          /* torch rounds the scalar to the tensor's fp32 */
    for (t = B - 1; t >= 0; --t) {
        float delta = r[t] + g32 * (1.0f - dw[t]) * vs_next[t] - vs[t];                 /* :203 (torch fp32) */
        gae = delta + gl * gae * (1.0f - done[t]);                                      /* :205 */
        adv[t] = gae;                                                                   /* :206 */
        v_target[t] = gae + vs[t];                                                      /* :208 */
    }
}
void orc_adv_normalize(float* adv, int64_t B) {             /* :210, torch mean / unbiased std */
    double s = 0, ss = 0, mean, var;
    int64_t t;
    for (t = 0; t < B; ++t) s += adv[t];
    mean = s / (double)B;
    for (t = 0; t < B; ++t) { double d = adv[t] - mean; ss += d * d; }
    var = ss / (double)(B - 1);
    for (t = 0; t < B; ++t) adv[t] = (float)((adv[t] - (float)mean) / ((float)sqrt(var) + 1e-5f));
}

/* ------------------------------------------------------------------------------------------
 * Actor_Gaussian / Critic forward, ppo_continuous.py:83-95, 123-128 (tanh activations), fp32
 * ------------------------------------------------------------------------------------------ */
static void mlp2(const float* W1, const float* b1, const float* W2, const float* b2,
                 int in_dim, int hid, const float* s, float* h2) {
    float* h1 = (float*)malloc(sizeof(float) * hid);
    int j, k;
    for (j = 0; j < hid; ++j) {
        float acc = b1[j];
        for (k = 0; k < in_dim; ++k) acc += W1[j * in_dim + k] * s[k];
        h1[j] = tanhf(acc);
    }
    for (j = 0; j < hid; ++j) {
        float acc = b2[j];
        for (k = 0; k < hid; ++k) acc += W2[j * hid + k] * h1[k];
        h2[j] = tanhf(acc);
    }
    free(h1);
}
void orc_actor_forward(const float* W1, const float* b1, const float* W2, const float* b2,
                       const float* W3, const float* b3, int in_dim, int hid, int act_dim,
                       float max_action, const float* s, int64_t n, float* mean) {
    int64_t i;
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
    for (i = 0; i < n; ++i) {
        float* h2 = (float*)malloc(sizeof(float) * hid);
        int j, k;
        mlp2(W1, b1, W2, b2, in_dim, hid, s + i * in_dim, h2);
        for (j = 0; j < act_dim; ++j) {
            float acc = b3[j];
            for (k = 0; k < hid; ++k) acc += W3[j * hid + k] * h2[k];
            mean[i * act_dim + j] = max_action * tanhf(acc);                             /* :87 */
        }
        free(h2);
    }
}
void orc_critic_forward(const float* W1, const float* b1, const float* W2, const float* b2,
                        const float* W3, const float* b3, int in_dim, int hid,
                        const float* s, int64_t n, float* v) {
    int64_t i;
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
    for (i = 0; i < n; ++i) {
        float* h2 = (float*)malloc(sizeof(float) * hid);
        float acc = b3[0];
        int k;
        mlp2(W1, b1, W2, b2, in_dim, hid, s + i * in_dim, h2);
        for (k = 0; k < hid; ++k) acc += W3[k] * h2[k];
        v[i] = acc;                                                                      /* :127 */
        free(h2);
    }
}
void orc_gaussian_sample(const float* mean, const float* log_std, const float* eps, int64_t n, int act_dim,
                         float max_action, float* a, float* logp) {
    /* :92-94 Normal(mean, exp(log_std)); :186 sample = mean + std*eps; :187 clamp; :188 log_prob */
    int64_t i;
    int j;
    for (i = 0; i < n; ++i)
        for (j = 0; j < act_dim; ++j) {
            float std = expf(log_std[j]);
            float m = mean[i * act_dim + j];
            float x = m + std * eps[i * act_dim + j];
            float var, lp;
            if (x < -max_action) x = -max_action;
            if (x > max_action) x = max_action;
            var = std * std;
            /* torch.distributions.Normal.log_prob: -((x-m)^2)/(2 var) - log(std) - log(sqrt(2 pi)) */
            lp = -((x - m) * (x - m)) / (2 * var) - logf(std) - 0.9189385332046727f;
            a[i * act_dim + j] = x; logp[i * act_dim + j] = lp;
        }
}

/* ------------------------------------------------------------------------------------------
 * Numerical_calculation_method.orbit_ode / numerical_calculation, satellite_function.py:793-839:
 * scipy.integrate.solve_ivp(method="RK45", rtol=1e-3, atol=1e-6, t_eval=arange(0, t+50, 50)) on the CW ODE,
 * value at the last t_eval point (= t_bound). Restates scipy 1.18.1's RungeKutta._step_impl, select_initial_step
 * and RkDenseOutput (third-party, Dormand-Prince 5(4)); w2 = 2*omega, w3 = 3*omega**2, wz = omega**2 are computed
 * by the caller exactly as python does (:801, :818-820). Thrust and J2 terms are identically zero there.
 * ------------------------------------------------------------------------------------------ */
static void cw_rhs(const double X[6], double w2, double w3, double wz, double f[6]) {
    f[0] = X[3]; f[1] = X[4]; f[2] = X[5];
    f[3] = ((w2 * X[4] + w3 * X[0]) + 0.0) + 0.0;           /* :818 */
    f[4] = ((-w2) * X[3] + 0.0) + 0.0;                      /* :819 */
    f[5] = ((-wz) * X[2] + 0.0) + 0.0;                      /* :820 */
}
static double rms6(const double x[6]) {
    double s = 0; int k;
    for (k = 0; k < 6; ++k) s += x[k] * x[k];
    return sqrt(s) / sqrt(6.0);
}
static const double RK45_A[6][5] = {{0, 0, 0, 0, 0}, {0.2, 0, 0, 0, 0}, {0.075, 0.225, 0, 0, 0},
    {0.9777777777777777, -3.7333333333333334, 3.5555555555555554, 0, 0},
    {2.9525986892242035, -11.595793324188385, 9.822892851699436, -0.2908093278463649, 0},
    {2.8462752525252526, -10.757575757575758, 8.906422717743473, 0.2784090909090909, -0.2735313036020583}};
static const double RK45_B[6] = {0.09114583333333333, 0.0, 0.44923629829290207, 0.6510416666666666, -0.322376179245283, 0.13095238095238096};
static const double RK45_E[7] = {-0.0012326388888888888, 0.0, 0.0042527702905061394, -0.03697916666666667, 0.05086379716981132, -0.0419047619047619, 0.025};
static const double RK45_P[7][4] = {{1.0, -2.8535800653862835, 3.0717434641059005, -1.1270175653862835}, {0, 0, 0, 0},
    {0.0, 4.023133379230305, -6.249321565289, 2.675424484351598}, {0.0, -3.7324019615885042, 10.068970589843675, -5.685526961588504},
    {0.0, 2.5548038301849423, -6.399112377351017, 3.5219323679207912}, {0.0, -1.3744241142186024, 3.272657752246729, -1.7672812570757455},
    {0.0, 1.3824689317781436, -3.764937863556287, 2.382468931778144}};

int orc_cw_ode_rk45(double y[6], double t_bound, double w2, double w3, double wz, int* nsteps_out) {
    const double rtol = 1e-3, atol = 1e-6, SAFETY = 0.9, MIN_FACTOR = 0.2, MAX_FACTOR = 10.0, err_exp = -0.2;
    double t = 0.0, f[6], K[7][6], y_new[6], f_new[6], y_old[6], scale[6], tmp[6], h_abs, h = 0.0;
    int k, s, j, nsteps = 0;
    cw_rhs(y, w2, w3, wz, f);
    {   /* select_initial_step */
        double d0, d1, d2, h0, h1, y1[6], f1[6];
        for (k = 0; k < 6; ++k) scale[k] = atol + fabs(y[k]) * rtol;
        for (k = 0; k < 6; ++k) tmp[k] = y[k] / scale[k];
        d0 = rms6(tmp);
        for (k = 0; k < 6; ++k) tmp[k] = f[k] / scale[k];
        d1 = rms6(tmp);
        h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        h0 = fmin(h0, fabs(t_bound));
        for (k = 0; k < 6; ++k) y1[k] = y[k] + h0 * 1.0 * f[k];
        cw_rhs(y1, w2, w3, wz, f1);
        for (k = 0; k < 6; ++k) tmp[k] = (f1[k] - f[k]) / scale[k];
        d2 = rms6(tmp) / h0;
        if (d1 <= 1e-15 && d2 <= 1e-15) h1 = fmax(1e-6, h0 * 1e-3);
        else h1 = pow(0.01 / fmax(d1, d2), 1.0 / 5.0);
        h_abs = fmin(fmin(100 * h0, h1), fabs(t_bound));
    }
    while (t != t_bound) {                                   /* OdeSolver.step until finished */
        double min_step = 10 * fabs(nextafter(t, INFINITY) - t), t_new = t, error_norm;
        int accepted = 0, rejected = 0;
        if (h_abs < min_step) h_abs = min_step;
        while (!accepted) {
            if (h_abs < min_step) return -1;                 /* TOO_SMALL_STEP */
            h = h_abs; t_new = t + h;
            if (t_new - t_bound > 0) t_new = t_bound;
            h = t_new - t; h_abs = fabs(h);
            for (k = 0; k < 6; ++k) K[0][k] = f[k];           /* rk_step */
            for (s = 1; s < 6; ++s) {
                double ys[6];
                for (k = 0; k < 6; ++k) {
                    double dy = 0;
                    for (j = 0; j < s; ++j) dy += K[j][k] * RK45_A[s][j];
                    ys[k] = y[k] + dy * h;
                }
                cw_rhs(ys, w2, w3, wz, K[s]);
            }
            for (k = 0; k < 6; ++k) {
                double acc = 0;
                for (j = 0; j < 6; ++j) acc += K[j][k] * RK45_B[j];
                y_new[k] = y[k] + h * acc;
            }
            cw_rhs(y_new, w2, w3, wz, f_new);
            for (k = 0; k < 6; ++k) K[6][k] = f_new[k];
            for (k = 0; k < 6; ++k) {
                double e = 0;
                for (j = 0; j < 7; ++j) e += K[j][k] * RK45_E[j];
                scale[k] = atol + fmax(fabs(y[k]), fabs(y_new[k])) * rtol;
                tmp[k] = (e * h) / scale[k];
            }
            error_norm = rms6(tmp);
            if (error_norm < 1) {
                double factor = (error_norm == 0) ? MAX_FACTOR : fmin(MAX_FACTOR, SAFETY * pow(error_norm, err_exp));
                if (rejected) factor = fmin(1.0, factor);
                h_abs *= factor; accepted = 1;
            } else { h_abs *= fmax(MIN_FACTOR, SAFETY * pow(error_norm, err_exp)); rejected = 1; }
        }
        for (k = 0; k < 6; ++k) { y_old[k] = y[k]; y[k] = y_new[k]; f[k] = f_new[k]; }
        t = t_new; ++nsteps;
    }
    /* value at t_eval[-1] == t_bound comes from the dense output of the last step at x = 1 (ivp.py) */
    for (k = 0; k < 6; ++k) {
        double q = 0;
        for (j = 0; j < 4; ++j) { double c = 0; for (s = 0; s < 7; ++s) c += K[s][k] * RK45_P[s][j]; q += c; }
        y[k] = h * q + y_old[k];
    }
    if (nsteps_out) *nsteps_out = nsteps;
    return 0;
}

/* ------------------------------------------------------------------------------------------
 * Reachable-domain sweep, single_pluse_model/RD_single_pulse.py:40-148 (Reachable_Domain, N1 = 1): for every direction
 * (gama_i, alpha_j), i <= N2, j <= N3, the reachability test and the two fsolve extremes. Output order = the reference's
 * append order (i major, j minor); valid[i*(N3+1)+j] marks the directions the reference appends.
 * ------------------------------------------------------------------------------------------ */
void orc_reachable_domain(const double el[6], double delta_max, int N2, int N3, double u,
                          double* rf_max_xyz, double* rf_min_xyz, uint8_t* valid) {
    double a = el[0], e0 = el[1], f = el[5];
    double r0 = a * (1 - SQ(e0)) / (1 + e0 * cos(f));                          /* :47 */
    double p0 = a * (1 - SQ(e0));                                              /* :48 */
    double Delta_V = -delta_max + 2 * delta_max * 1 / 1;                       /* :65, N1 = 1 */
    int i, j;
    for (i = 0; i <= N2; ++i) {
        double gama = 2 * ORC_PI * i / N2;                                     /* :67 */
        for (j = 0; j <= N3; ++j) {
            double alpha = -ORC_PI / 2 + ORC_PI * j / N3;                      /* :69 */
            double P[3] = {sin(gama) * cos(alpha), cos(gama) * cos(alpha), sin(alpha)};   /* :72 */
            double temp1 = SQ(sin(gama - f)) / (u * SQ(1 + e0 * cos(f)) / (p0 * SQ(Delta_V)) - 1);   /* :80 */
            double t2 = SQ(tan(alpha));
            int64_t o = (int64_t)i * (N3 + 1) + j;
            int k;
            valid[o] = 0;
            for (k = 0; k < 3; ++k) { rf_max_xyz[o * 3 + k] = 0; rf_min_xyz[o * 3 + k] = 0; }
            if (0 <= t2 && t2 <= temp1) {                                      /* :82 */
                double beta = atan(tan(alpha) / sin(gama - f));                /* :83 */
                double Delta_Vm = sqrt(SQ(Delta_V) - u * SQ(1 + e0 * cos(f)) * SQ(sin(beta)) / p0);   /* :85 */
                double df = gama - f, theta = 0, rf[2], lo, hi;
                int g, have = 0;
                if ((-2 * ORC_PI <= df && df < -ORC_PI) || (0 <= df && df < ORC_PI)) { theta = acos(cos(df) * cos(alpha)); have = 1; }   /* :88-89 */
                else if ((-ORC_PI <= df && df < 0) || (ORC_PI <= df && df < 2 * ORC_PI)) { theta = 2 * ORC_PI - acos(cos(df) * cos(alpha)); have = 1; }
                (void)have;   /* outside both ranges python keeps theta from the previous direction; gama - f stays inside for f in [0, 2pi) */
                for (g = 0; g < 2; ++g) {
                    double ag = g == 0 ? ORC_PI / 2 : -ORC_PI / 2;             /* :94 / :109 */
                    double v_1x = sqrt(u / p0) * e0 * sin(f) + Delta_Vm * cos(ag);
                    double v_1y = sqrt(u / p0) * (1 + e0 * cos(f)) * cos(beta) + Delta_Vm * sin(ag);
                    double h = r0 * v_1y;
                    double al = orc_numerical_iteration(u, Delta_Vm, theta, v_1x, v_1y, h, ag);
                    double vx = sqrt(u / p0) * e0 * sin(f) + Delta_Vm * cos(al);
                    double vy = sqrt(u / p0) * (1 + e0 * cos(f)) * cos(beta) + Delta_Vm * sin(al);
                    double hm = r0 * vy;
                    rf[g] = SQ(hm) / (u * (1 - cos(theta)) + hm * vy * cos(theta) - hm * vx * sin(theta));   /* :107 / :121 */
                }
                hi = fmax(fabs(rf[0]), fabs(rf[1])); lo = fmin(fabs(rf[0]), fabs(rf[1]));   /* :123-124 */
                for (k = 0; k < 3; ++k) { rf_max_xyz[o * 3 + k] = hi * P[k]; rf_min_xyz[o * 3 + k] = lo * P[k]; }
                valid[o] = 1;
            }
        }
    }
}
