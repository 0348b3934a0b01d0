// glibm.cuh -- sin / cos / acos / atan / pow(x, 2) / pow(x, 0.5) with the SAME BITS as the host libm the reference runs on.
//
// Why this exists (DESIGN.md s3, VERDICT r01 item 1): the reference's danger-zone count
// (environment.py:317-332 -> satellite_function.py:161-255, :317-373, :462-565) is an integer that depends on the last
// bit of numpy scalar sin/cos/arccos/arctan and of python's `x ** 2` (= libm pow(x, 2.0)): scipy's fsolve takes a
// forward-difference Jacobian at +-pi/2 and a one-ulp change of sin(alpha) sends the Newton step to another branch of
// the root.  CUDA's libdevice differs from glibc in the last ulp of ~10 % of the calls, which flipped 3.2e-5 of the
// counts in round 1.  Correct rounding would not help either: glibc itself is only faithful (0.50x - 0.56 ulp), so the
// one way to get the reference's integer is to perform glibc's arithmetic.
//
// What is restated: GNU libm 2.39, sysdeps/ieee754/dbl-64 (third-party dependency of the reference, not part of the
// upstream repository; the version is the one of this image, Ubuntu GLIBC 2.39-0ubuntu8.5, x86-64):
//   s_sin.c   __sin / __cos   (do_sin, do_cos, TAYLOR_SIN, reduce_sincos; |x| < 105414350, above that -> NaN here)
//   e_asin.c  __ieee754_acos  (all ranges)
//   s_atan.c  __atan          (all ranges)
//   e_pow.c   __pow           (log_inline + exp_inline, for y == 2.0 and y == 0.5; y == 2: |x| outside [2^-369, 2^369] -> x*x here)
// in the variant the ifunc resolvers select on every FMA-capable x86-64 host (__sin_fma, __cos_fma, __atan_fma,
// __ieee754_acos_fma, __pow_fma): those are the generic sources compiled with -mfma, i.e. with GCC's contraction of
// a*b+c into fused operations.  Which operations are fused was read off the machine code of the libm in this image;
// every fused operation is spelled fma_() below and everything else is an individually rounded mul_/add_/sub_, so
// the result does not depend on this file's own compiler flags.  The lookup tables are glibc's (glibm_tables.inc).
// numpy's float64 arccos/arctan call libm on hosts without AVX-512 and an SVML-derived kernel with different last
// bits on AVX-512 hosts, so "the reference" is host dependent there; the CPU oracle (glibc) is the pinned variant.
//
// Verified bit for bit against the real libm on the host (the same header compiles with g++):
// tests/test_glibm_host.py (every CPU test run) and tools/soak_glibm.py (1e9-sample soak).
#pragma once
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define GLIBM_FN __device__ __forceinline__
#define GLIBM_FN_NOINLINE __device__ __noinline__
#define GLIBM_TABLE static __device__ const
#else
#include <cmath>
#define GLIBM_FN static inline
#define GLIBM_FN_NOINLINE static inline
#define GLIBM_TABLE static const
#endif

#include "glibm_tables.inc"

namespace glibm {

// individually rounded IEEE operations (no contraction whatever the flags) and the spelled fused one
#if defined(__CUDACC__)
GLIBM_FN double mul_(double a, double b) { return __dmul_rn(a, b); }
GLIBM_FN double add_(double a, double b) { return __dadd_rn(a, b); }
GLIBM_FN double sub_(double a, double b) { return __dsub_rn(a, b); }
GLIBM_FN double div_(double a, double b) { return __ddiv_rn(a, b); }
GLIBM_FN double fma_(double a, double b, double c) { return __fma_rn(a, b, c); }
GLIBM_FN uint64_t bits_(double x) { return (uint64_t)__double_as_longlong(x); }
GLIBM_FN double dbl_(uint64_t u) { return __longlong_as_double((long long)u); }
GLIBM_FN double abs_(double x) { return fabs(x); }
GLIBM_FN double nan_() { return __longlong_as_double(0x7ff8000000000000ll); }
#else
GLIBM_FN double mul_(double a, double b) { volatile double r = a * b; return r; }
GLIBM_FN double add_(double a, double b) { volatile double r = a + b; return r; }
GLIBM_FN double sub_(double a, double b) { volatile double r = a - b; return r; }
GLIBM_FN double div_(double a, double b) { volatile double r = a / b; return r; }
GLIBM_FN double fma_(double a, double b, double c) { return __builtin_fma(a, b, c); }
GLIBM_FN uint64_t bits_(double x) { uint64_t u; std::memcpy(&u, &x, 8); return u; }
GLIBM_FN double dbl_(uint64_t u) { double x; std::memcpy(&x, &u, 8); return x; }
GLIBM_FN double abs_(double x) { return __builtin_fabs(x); }
GLIBM_FN double nan_() { return __builtin_nan(""); }
#endif
GLIBM_FN double neg_(double x) { return dbl_(bits_(x) ^ 0x8000000000000000ull); }
GLIBM_FN double copysign_(double mag, double sgn) {
    return dbl_((bits_(mag) & 0x7fffffffffffffffull) | (bits_(sgn) & 0x8000000000000000ull));
}
GLIBM_FN int32_t hi32_(double x) { return (int32_t)(bits_(x) >> 32); }
GLIBM_FN uint32_t lo32_(double x) { return (uint32_t)bits_(x); }

// ---------------------------------------------------------------------------------------------------------------
// s_sin.c
// ---------------------------------------------------------------------------------------------------------------
namespace k {
constexpr double BIG = 0x1.8p45, TOINT = 0x1.8p52, HPINV = 0x1.45f306dc9c883p-1;
constexpr double MP1 = 0x1.921fb58p+0, MP2 = -0x1.dde973cp-27, PP3 = -0x1.cb3b398p-55, PP4 = -0x1.d747f23e32ed7p-83;
constexpr double HP0 = 0x1.921fb54442d18p+0, HP1 = 0x1.1a62633145c07p-54, PI = 0x1.921fb54442d18p+1;
constexpr double SN3 = -0x1.5555555555515p-3, SN5 = 0x1.11110e829872fp-7;
constexpr double CS2 = 0.5, CS4 = -0x1.5555555555535p-5, CS6 = 0x1.6c16bedd9e239p-10;
constexpr double S1 = -0x1.5555555555555p-3, S2 = 0x1.1111111110ecep-7, S3 = -0x1.a01a019db08b8p-13,
                 S4 = 0x1.71de27b9a7ed9p-19, S5 = -0x1.addffc2fcdf59p-26;
}  // namespace k

// TAYLOR_SIN (xx = x*x): x + ((POLY(xx) x - dx/2) xx + dx)
GLIBM_FN double taylor_sin(double x, double dx) {
    const double xx = mul_(x, x);
    double p = k::S5;
    p = fma_(p, xx, k::S4); p = fma_(p, xx, k::S3); p = fma_(p, xx, k::S2); p = fma_(p, xx, k::S1);
    const double t = fma_(p, x, neg_(mul_(dx, 0.5)));
    return add_(x, fma_(xx, t, dx));
}

// the table step shared by do_sin / do_cos: u = BIG + |x| rounds |x| to a multiple of 1/128 (table index in the low
// mantissa bits); returns the remainder |x| - k/128
GLIBM_FN double tab_split(double ax, int& idx) {
    const double u = add_(k::BIG, ax);
    idx = (int)(lo32_(u) << 2);
    return sub_(ax, sub_(u, k::BIG));
}

// sin(x + dx) for |x| < 0.855469 + (reduction slack)
GLIBM_FN double do_sin(double x, double dx) {
    if (abs_(x) < 0.126) return taylor_sin(x, dx);
    if (x <= 0.0) dx = neg_(dx);
    int i;
    const double xr = tab_split(abs_(x), i);
    const double xx = mul_(xr, xr);
    const double s = add_(xr, fma_(mul_(xr, xx), fma_(k::SN5, xx, k::SN3), dx));
    const double c = fma_(xr, dx, mul_(xx, fma_(fma_(k::CS6, xx, k::CS4), xx, k::CS2)));
    const double sn = glibm_sincos[i], ssn = glibm_sincos[i + 1], cs = glibm_sincos[i + 2], ccs = glibm_sincos[i + 3];
    const double cor = fma_(s, cs, fma_(neg_(c), sn, fma_(s, ccs, ssn)));
    return copysign_(add_(sn, cor), x);
}

// cos(x + dx), same range
GLIBM_FN double do_cos(double x, double dx) {
    if (x < 0.0) dx = neg_(dx);
    int i;
    const double xr = add_(tab_split(abs_(x), i), dx);
    const double xx = mul_(xr, xr);
    const double s = fma_(mul_(xr, xx), fma_(k::SN5, xx, k::SN3), xr);
    const double c = mul_(xx, fma_(fma_(k::CS6, xx, k::CS4), xx, k::CS2));
    const double sn = glibm_sincos[i], ssn = glibm_sincos[i + 1], cs = glibm_sincos[i + 2], ccs = glibm_sincos[i + 3];
    const double cor = fma_(neg_(s), sn, fma_(neg_(c), cs, fma_(neg_(s), ssn, ccs)));
    return add_(cs, cor);
}

// reduce_sincos: x = n pi/2 + (a + da), 2.426265 < |x| < 105414350; returns n & 3
GLIBM_FN int reduce_sincos(double x, double& a, double& da) {
    const double t = fma_(x, k::HPINV, k::TOINT);
    const double xn = sub_(t, k::TOINT);
    const int n = (int)(lo32_(t) & 3u);
    const double y = fma_(neg_(xn), k::MP2, fma_(neg_(xn), k::MP1, x));
    const double t2 = fma_(neg_(xn), k::PP3, y);
    const double db = fma_(neg_(k::PP3), xn, sub_(y, t2));
    const double b = fma_(neg_(xn), k::PP4, t2);
    const double db2 = fma_(neg_(xn), k::PP4, sub_(t2, b));
    a = b;
    da = add_(db, db2);
    return n;
}

GLIBM_FN double do_sincos(double a, double da, int n) {
    const double r = (n & 1) ? do_cos(a, da) : do_sin(a, da);
    return (n & 2) ? neg_(r) : r;
}

GLIBM_FN double sin(double x) {
    const int32_t kk = hi32_(x) & 0x7fffffff;
    if (kk < 0x3e500000) return x;                                           // |x| < 2^-26
    if (kk < 0x3feb6000) return do_sin(x, 0.0);                              // |x| < 0.855469
    if (kk < 0x400368fd) return copysign_(do_cos(sub_(k::HP0, abs_(x)), k::HP1), x);   // |x| < 2.426265
    if (kk < 0x419921fb) { double a, da; const int n = reduce_sincos(x, a, da); return do_sincos(a, da, n); }
    return nan_();                                                           // glibc: __branred (not restated) / inf, nan
}

GLIBM_FN double cos(double x) {
    const int32_t kk = hi32_(x) & 0x7fffffff;
    if (kk < 0x3e400000) return 1.0;                                         // |x| < 2^-27
    if (kk < 0x3feb6000) return do_cos(x, 0.0);
    if (kk < 0x400368fd) {
        const double y = sub_(k::HP0, abs_(x));
        const double a = add_(y, k::HP1);
        return do_sin(a, add_(sub_(y, a), k::HP1));
    }
    if (kk < 0x419921fb) { double a, da; const int n = reduce_sincos(x, a, da); return do_sincos(a, da, n + 1); }
    return nan_();
}

// both at once; the range reduction (the only shareable part) is done once. Same bits as sin(x), cos(x).
// Written so that a warp whose lanes sit in different ranges still runs ONE do_sin and ONE do_cos evaluation: every
// range of __sin and __cos above 2^-26 is one call of each with range-dependent arguments.
GLIBM_FN void sincos(double x, double* s, double* c) {
    const int32_t kk = hi32_(x) & 0x7fffffff;
    if (kk < 0x3e500000 || kk >= 0x419921fb) { *s = sin(x); *c = cos(x); return; }      // tiny, huge, inf, nan
    double sa, sda, ca, cda;       // arguments of the do_sin call and of the do_cos call
    int n = 0;                     // quadrant: 0 -> (sin, cos) = (ds, dc); 1 -> (dc, -ds); 2 -> (-ds, -dc); 3 -> (-dc, ds)
    bool mid = false;
    if (kk < 0x3feb6000) { sa = x; sda = 0.0; ca = x; cda = 0.0; }
    else if (kk < 0x400368fd) {
        const double y = sub_(k::HP0, abs_(x));
        ca = y; cda = k::HP1;                                                // sin(x) = copysign(do_cos(y, hp1), x)
        sa = add_(y, k::HP1); sda = add_(sub_(y, sa), k::HP1);               // cos(x) = do_sin(a, da)
        mid = true;
    } else {
        n = reduce_sincos(x, sa, sda);
        ca = sa; cda = sda;
    }
    const double ds = do_sin(sa, sda), dc = do_cos(ca, cda);
    if (mid) { *s = copysign_(dc, x); *c = ds; return; }
    const double sv = (n & 1) ? dc : ds, cv = (n & 1) ? ds : dc;
    *s = (n & 2) ? neg_(sv) : sv;
    *c = ((n + 1) & 2) ? neg_(cv) : cv;
}

// ---------------------------------------------------------------------------------------------------------------
// e_asin.c: __ieee754_acos
// ---------------------------------------------------------------------------------------------------------------
namespace k {
constexpr double F1 = 0x1.55555555554f9p-3, F2 = 0x1.333333336127dp-4, F3 = 0x1.6db6dae42c0e4p-5, F4 = 0x1.f1c7e04f4ad99p-6,
                 F5 = 0x1.6e442c822d419p-6, F6 = 0x1.292d80f453c72p-6;
constexpr double RT0 = 0x1.fffffffecc1ddp-1, RT1 = 0x1.fffffff757304p-2, RT2 = 0x1.800496769c91ap-2, RT3 = 0x1.4006318d1dab9p-2;
constexpr double T27 = 0x1p27;
}  // namespace k

GLIBM_FN double asin_poly(double z) {      // (((((f6 z + f5) z + f4) z + f3) z + f2) z + f1)
    double p = k::F6;
    p = fma_(p, z, k::F5); p = fma_(p, z, k::F4); p = fma_(p, z, k::F3); p = fma_(p, z, k::F2); p = fma_(p, z, k::F1);
    return p;
}

// table ranges: ax = |x|, row at asncs[n] = {x_i, c1 .. c_deg, c_{deg+1}, asin(x_i) head, (unused here)}. The six ranges of
// e_asin.c differ only in the row width and the polynomial degree (6 .. 10), so they run through ONE code path: the Horner
// recurrence starts at degree 10 with p = 0 and zero coefficients above `deg` - fma(0, xx, 0) = 0 and fma(0, xx, c_deg) = c_deg
// exactly, so the bits are those of the degree-`deg` recurrence, and a warp whose lanes sit in different ranges does not
// execute six copies of the routine.
GLIBM_FN double acos_tab(double ax, int n, int deg, bool pos) {
    const double* T = glibm_asncs + n;
    const double xx = sub_(ax, T[0]);
    double p = 0.0;
#pragma unroll
    for (int j = 10; j >= 2; --j) p = fma_(p, xx, (j <= deg) ? T[j] : 0.0);
    p = fma_(p, mul_(xx, xx), T[deg + 1]);
    const double t = fma_(xx, T[1], p);
    const double y = T[deg + 2];
    return pos ? add_(sub_(k::HP1, t), sub_(k::HP0, y)) : add_(add_(t, k::HP1), add_(y, k::HP0));
}

GLIBM_FN double acos(double x) {
    const int32_t m = hi32_(x);
    const int32_t kk = m & 0x7fffffff;
    const bool pos = m > 0;
    if (kk < 0x3c880000) return k::HP0;                                      // |x| < 2^-55
    if (kk < 0x3fc00000) {                                                   // |x| < 0.125
        const double x2 = mul_(x, x);
        const double p = asin_poly(x2);
        const double r = sub_(k::HP0, x);
        const double c0 = add_(sub_(sub_(k::HP0, r), x), k::HP1);
        return add_(r, fma_(neg_(p), mul_(x, x2), c0));
    }
    const double ax = pos ? x : neg_(x);
    if (kk < 0x3fef0000) {                                                   // 0.125 <= |x| < 0.96875: the six table ranges
        const int i13 = (kk >> 13) & 0x7f;
        int n, deg;
        if (kk < 0x3fd00000) { n = 11 * ((kk >> 15) & 0x1f); deg = 6; }              // < 0.25
        else if (kk < 0x3fe00000) { n = 11 * ((kk >> 14) & 0x3f) + 352; deg = 6; }   // < 0.5
        else if (kk < 0x3fe80000) { n = 12 * i13 + 1056; deg = 7; }                  // < 0.75
        else if (kk < 0x3fed8000) { n = 13 * i13 + 992; deg = 8; }                   // < 0.921875
        else if (kk < 0x3fee8000) { n = 14 * i13 + 884; deg = 9; }                   // < 0.953125
        else { n = 15 * i13 + 768; deg = 10; }                                       // < 0.96875
        return acos_tab(ax, n, deg, pos);
    }
    if (kk < 0x3ff00000) {                                                   // < 1: acos = 2 asin(sqrt((1 - |x|) / 2))
        const double z = mul_(pos ? sub_(1.0, x) : add_(x, 1.0), 0.5);
        const uint64_t v = bits_(z);
        double t = mul_(glibm_inroot[(v >> 46) & 0x7f], glibm_powtwo[511 - (int)(v >> 53)]);
        const double r = fma_(neg_(mul_(t, t)), z, 1.0);
        double q = k::RT3;
        q = fma_(q, r, k::RT2); q = fma_(q, r, k::RT1); q = fma_(q, r, k::RT0);
        t = mul_(q, t);
        const double c = mul_(z, t);
        const double w = fma_(neg_(c), mul_(t, 0.5), 1.5);
        const double y = fma_(neg_(k::T27), c, fma_(c, k::T27, c));
        const double cc = div_(fma_(neg_(y), y, z), fma_(w, c, y));
        const double ps = mul_(mul_(asin_poly(z), z), add_(y, cc));
        double res;
        if (m < 0) res = add_(sub_(sub_(k::HP1, cc), ps), sub_(k::HP0, y));
        else res = add_(add_(cc, ps), y);
        return add_(res, res);
    }
    if (kk == 0x3ff00000 && lo32_(x) == 0u) return pos ? 0.0 : k::PI;        // |x| == 1
    return nan_();                                                           // |x| > 1 or NaN
}

// ---------------------------------------------------------------------------------------------------------------
// s_atan.c: __atan
// ---------------------------------------------------------------------------------------------------------------
namespace k {
constexpr double AT_A = 0x1.bb67ap-27, AT_B = 0x1p-4, AT_D = 16.0, AT_E = 0x1.49ff2p+52;
constexpr double D3 = -0x1.5555555555555p-2, D5 = 0x1.99999999997fdp-3, D7 = -0x1.24924923f7603p-3, D9 = 0x1.c71c6e5129a3bp-4,
                 D11 = -0x1.7458022b13c25p-4, D13 = 0x1.375f08b31cbcep-4;
constexpr double TWO52 = 0x1p52, TWO8 = 256.0;
}  // namespace k

GLIBM_FN double atan_poly(double v) {      // d3 + v (d5 + v (d7 + v (d9 + v (d11 + v d13))))
    double yy = k::D13;
    yy = fma_(yy, v, k::D11); yy = fma_(yy, v, k::D9); yy = fma_(yy, v, k::D7); yy = fma_(yy, v, k::D5); yy = fma_(yy, v, k::D3);
    return yy;
}
GLIBM_FN const double* atan_row(double u) {      // i = rint(256 u) - 16
    const int i = (int)sub_(fma_(u, k::TWO8, k::TWO52), k::TWO52) - 16;
    return glibm_cij + 7 * i;
}
GLIBM_FN double atan_row_poly(const double* C, double z) {   // c2 + z (c3 + z (c4 + z (c5 + z c6)))
    double yy = C[6];
    yy = fma_(yy, z, C[5]); yy = fma_(yy, z, C[4]); yy = fma_(yy, z, C[3]); yy = fma_(yy, z, C[2]);
    return yy;
}

GLIBM_FN double atan(double x) {
    if (x != x) return add_(x, x);
    const double u = abs_(x);
    if (u < 1.0) {
        if (u < k::AT_B) {
            if (u < k::AT_A) return x;
            const double v = mul_(x, x);
            return fma_(mul_(x, v), atan_poly(v), x);
        }
        const double* C = atan_row(u);
        const double z = sub_(u, C[0]);
        return copysign_(fma_(atan_row_poly(C, z), z, C[1]), x);
    }
    if (u < k::AT_D) {
        const double w = div_(1.0, u);
        const double t1 = mul_(w, u);
        const double t2 = fma_(u, w, neg_(t1));
        const double e = sub_(sub_(1.0, t1), t2);
        const double* C = atan_row(w);
        const double z = fma_(e, w, sub_(w, C[0]));
        const double yy = fma_(neg_(atan_row_poly(C, z)), z, k::HP1);
        return copysign_(add_(sub_(k::HP0, C[1]), yy), x);
    }
    if (u < k::AT_E) {
        const double w = div_(1.0, u);
        const double t1 = mul_(w, u);
        const double t3 = sub_(k::HP0, w);
        const double v = mul_(w, w);
        const double yy = atan_poly(v);
        const double cor = add_(sub_(sub_(k::HP0, t3), w), k::HP1);
        const double t2 = fma_(u, w, neg_(t1));
        const double e = sub_(sub_(1.0, t1), t2);
        const double a = fma_(neg_(e), w, cor);
        const double b = fma_(neg_(mul_(w, v)), yy, a);
        return copysign_(add_(t3, b), x);
    }
    return copysign_(k::HP0, x);
}

// ---------------------------------------------------------------------------------------------------------------
// e_pow.c: pow(x, 2.0)  (python / numpy scalar `x ** 2`) and pow(x, 0.5)
// ---------------------------------------------------------------------------------------------------------------
namespace k {
constexpr double LN2HI = 0x1.62e42fefa3800p-1, LN2LO = 0x1.ef35793c76730p-45;
constexpr double A0 = -0x1p-1, A1 = -0x1.5555555555560p-1, A2 = 0x1.0000000000006p-1, A3 = 0x1.999999959554ep-1,
                 A4 = -0x1.555555529a47ap-1, A5 = -0x1.2495b9b4845e9p+0, A6 = 0x1.0002b8b263fc3p+0;
constexpr double INVLN2N = 0x1.71547652b82fep+7, SHIFT = 0x1.8p52, NEGLN2HIN = -0x1.62e42fefa0000p-8, NEGLN2LON = -0x1.cf79abc9e3b3ap-47;
constexpr double C2 = 0x1.ffffffffffdbdp-2, C3 = 0x1.555555555543cp-3, C4 = 0x1.55555cf172b91p-5, C5 = 0x1.1111167a4d017p-7;
}  // namespace k

// log_inline + exp_inline of e_pow.c for y = 2 or 0.5: ix is the bit pattern of a positive normal x whose |y log x| stays
// below 512, so neither of exp_inline's special cases is reached
GLIBM_FN double pow_core(uint64_t ix, double y) {
    // log_inline
    const uint64_t tmp = ix - 0x3fe6955500000000ull;
    const int i = (int)((tmp >> 45) & 0x7f);
    const int kexp = (int)((int64_t)tmp >> 52);
    const double z = dbl_(ix - (tmp & 0xfff0000000000000ull));
    const double kd = (double)kexp;
    const double invc = glibm_powlog[3 * i], logc = glibm_powlog[3 * i + 1], logctail = glibm_powlog[3 * i + 2];
    const double r = fma_(z, invc, -1.0);
    const double t1 = fma_(kd, k::LN2HI, logc);
    const double t2 = add_(t1, r);
    const double lo1 = fma_(kd, k::LN2LO, logctail);
    const double lo2 = add_(sub_(t1, t2), r);
    const double ar = mul_(k::A0, r);
    const double ar2 = mul_(r, ar);
    const double ar3 = mul_(r, ar2);
    const double hi = add_(t2, ar2);
    const double lo3 = fma_(ar, r, neg_(ar2));
    const double lo4 = add_(sub_(t2, hi), ar2);
    const double p12 = fma_(k::A2, r, k::A1), p34 = fma_(k::A4, r, k::A3), p56 = fma_(k::A6, r, k::A5);
    const double pp = fma_(ar2, fma_(p56, ar2, p34), p12);
    const double lo = fma_(ar3, pp, add_(add_(add_(lo1, lo2), lo3), lo4));
    const double lhi = add_(hi, lo);
    const double llo = add_(sub_(hi, lhi), lo);
    // pow: ehi + elo = y log(x)
    const double ehi = mul_(y, lhi);
    const double elo = fma_(y, llo, fma_(lhi, y, neg_(ehi)));
    // exp_inline
    const uint32_t abstop = (uint32_t)(bits_(ehi) >> 52) & 0x7ffu;
    if (abstop < 0x3c9u) return add_(1.0, ehi);                              // |y log x| < 2^-54
    const double kdz = fma_(ehi, k::INVLN2N, k::SHIFT);
    const uint64_t ki = bits_(kdz);
    const double kd2 = sub_(kdz, k::SHIFT);
    double rr = fma_(kd2, k::NEGLN2LON, fma_(kd2, k::NEGLN2HIN, ehi));
    rr = add_(elo, rr);
    const int idx = 2 * (int)(ki & 0x7f);
    const double tail = dbl_(glibm_exptab[idx]);
    const uint64_t sbits = glibm_exptab[idx + 1] + (ki << 45);
    const double r2 = mul_(rr, rr);
    const double q23 = fma_(k::C3, rr, k::C2), q45 = fma_(rr, k::C5, k::C4);
    const double tmp2 = fma_(q45, mul_(r2, r2), fma_(q23, r2, add_(rr, tail)));
    const double scale = dbl_(sbits);
    return fma_(tmp2, scale, scale);
}

GLIBM_FN double pow2(double x) {
    uint64_t ix = bits_(x) & 0x7fffffffffffffffull;                          // y = 2 is an even integer: sign of x is dropped
    uint32_t topx = (uint32_t)(ix >> 52);
    if (topx == 0x7ffu || ix == 0ull) return mul_(x, x);                     // 0, inf, nan
    if (topx == 0u) { ix = (bits_(mul_(dbl_(ix), 0x1p52)) & 0x7fffffffffffffffull) - (52ull << 52); topx = (uint32_t)(ix >> 52) & 0x7ffu; }
    if (topx < 0x3ffu - 369u || topx > 0x3ffu + 369u) return mul_(x, x);     // result near over/underflow: not restated
    return pow_core(ix, 2.0);
}

// pow(x, 0.5) (python `x ** 0.5`; not sqrt(x): glibc's pow is not correctly rounded). |0.5 log x| < 373 for every positive
// double, so all of them are restated.
GLIBM_FN double pow_half(double x) {
    uint64_t ix = bits_(x);
    if (2 * ix - 1 >= 2 * 0x7ff0000000000000ull - 1) return mul_(x, x);     // +-0, +-inf, nan (e_pow.c zeroinfnan)
    if (ix >> 63) return nan_();                                             // finite x < 0: invalid
    if ((ix >> 52) == 0u) ix = (bits_(mul_(x, 0x1p52)) & 0x7fffffffffffffffull) - (52ull << 52);   // subnormal
    return pow_core(ix, 0.5);
}

#if defined(__CUDACC__)
// Out-of-line copies for straight-line device code with many call sites (orbital elements, danger-zone set-up): one
// body per function keeps the kernel inside the instruction cache (inlined everywhere the danger-zone kernel grew to
// 15 000 SASS instructions and stalled on instruction fetch). Results come back in registers.
namespace call {
static __device__ __noinline__ double2 sincos(double x) { double s, c; glibm::sincos(x, &s, &c); return make_double2(s, c); }
static __device__ __noinline__ double cos(double x) { return glibm::cos(x); }
static __device__ __noinline__ double acos(double x) { return glibm::acos(x); }
static __device__ __noinline__ double atan(double x) { return glibm::atan(x); }
static __device__ __noinline__ double pow2(double x) { return glibm::pow2(x); }
static __device__ __noinline__ double pow_half(double x) { return glibm::pow_half(x); }
}  // namespace call
#endif

}  // namespace glibm
