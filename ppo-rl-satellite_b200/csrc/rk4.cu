// rk4.cu -- K1: batched fp64 RK4 two-body(+J2) propagator for sm_100a, plus the DFMA/FFMA peak probes.
//
// Reference behaviour replaced: StateEq + RungeKutta ("轨道外推-龙格库塔算法.py":15-40), called
// `substeps` times per state. One thread integrates ILP independent states held in registers for all
// substeps; HBM is touched once on entry and once on exit (96 B per state per launch), so the kernel
// is FP64-pipe bound for substeps >= 4 and HBM/launch bound below that.
//
// Layout: SoA x[6][ld] (rows x,y,z,vx,vy,vz). With ILP = 2 each thread owns two adjacent states and
// moves them with 128-bit ld/st.global.v2.f64 (ld even, base 16-byte aligned).
#include "sat_math.cuh"
#include "../../include/satb200.h"

namespace {
using namespace sat;

constexpr int kThreads = 128;

template <bool J2, int ILP>
__global__ void __launch_bounds__(kThreads)
rk4_kernel(double* __restrict__ x, int64_t n, int64_t ld, int substeps, double h, double mu, double re, double j2) {
    const int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    const int64_t i0 = t * ILP;
    if (i0 >= n) return;
    const Rk4Consts c = make_rk4_consts(h, mu, re, j2);
    double r[ILP][3], v[ILP][3];
    const bool full = (i0 + ILP <= n);
    if (ILP == 2 && full) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double2 a = *reinterpret_cast<const double2*>(x + k * ld + i0);
            double2 b = *reinterpret_cast<const double2*>(x + (3 + k) * ld + i0);
            r[0][k] = a.x; r[ILP - 1][k] = a.y; v[0][k] = b.x; v[ILP - 1][k] = b.y;
        }
    } else {
#pragma unroll
        for (int j = 0; j < ILP; ++j) {
            const int64_t i = (i0 + j < n) ? i0 + j : i0;
#pragma unroll
            for (int k = 0; k < 3; ++k) { r[j][k] = x[k * ld + i]; v[j][k] = x[(3 + k) * ld + i]; }
        }
    }
#pragma unroll 1
    for (int s = 0; s < substeps; ++s) {
#pragma unroll
        for (int j = 0; j < ILP; ++j) rk4_step<J2>(r[j], v[j], c);
    }
    if (ILP == 2 && full) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            *reinterpret_cast<double2*>(x + k * ld + i0) = make_double2(r[0][k], r[ILP - 1][k]);
            *reinterpret_cast<double2*>(x + (3 + k) * ld + i0) = make_double2(v[0][k], v[ILP - 1][k]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < ILP; ++j) {
            if (i0 + j < n) {
#pragma unroll
                for (int k = 0; k < 3; ++k) { x[k * ld + i0 + j] = r[j][k]; x[(3 + k) * ld + i0 + j] = v[j][k]; }
            }
        }
    }
}

template <typename T>
__global__ void peak_kernel(T* sink, int iters) {
    // 16 independent FMA chains per thread: enough ILP to saturate the pipe at any occupancy
    T a[16];
    const T m = (T)1.0000001, c = (T)1e-7;
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = (T)(threadIdx.x + k) * (T)1e-3;
    // unrolled x8: 128 FMAs per loop-overhead triple (add / compare / branch). With `unroll 1` the three overhead instructions
    // took 3 of 19 issue slots and the "peak" read 85 % of the pipe rate (round-1 finding)
#pragma unroll 8
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k] = fma(a[k], m, c);
    }
    T s = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += a[k];
    if (s == (T)-1.2345) sink[0] = s;     // never true; keeps the chains alive
}


// ------------------------------------------------------------------------------------------------
// helper kernels behind the satellite_function.py facade (batched forms of the reference helpers)
// ------------------------------------------------------------------------------------------------
// StateEq (script :15-30): f = [v, a(x)]
template <bool J2>
__global__ void state_eq_kernel(const double* __restrict__ x, double* __restrict__ f, int64_t n, int64_t ld,
                                double mu, double re, double j2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double ax, ay, az;
    accel_scaled<J2>(x[i], x[ld + i], x[2 * ld + i], 1.5 * j2 * re * re, ax, ay, az);
    f[i] = x[3 * ld + i]; f[ld + i] = x[4 * ld + i]; f[2 * ld + i] = x[5 * ld + i];
    f[3 * ld + i] = -mu * ax; f[4 * ld + i] = -mu * ay; f[5 * ld + i] = -mu * az;
}

// Clohessy_Wiltshire.State_transition_matrix (satellite_function.py:753-781): x <- M x, numpy's dgemv order
struct Stm36 { double m[36]; };
__global__ void cw_apply_kernel(double* __restrict__ x, int64_t n, int64_t ld, const __grid_constant__ Stm36 M) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double v[6], y[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) v[k] = x[k * ld + i];
#pragma unroll
    for (int k = 0; k < 6; ++k) y[k] = gemv6_row(M.m + 6 * k, v);
#pragma unroll
    for (int k = 0; k < 6; ++k) x[k * ld + i] = y[k];
}

// calculate_orbital_elements (satellite_function.py:161-255), six-element branch
__global__ void elements_kernel(const double* __restrict__ rv, int64_t n, double miu, double* __restrict__ out,
                                int32_t* __restrict__ kind) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double R[3] = {rv[i * 6], rv[i * 6 + 1], rv[i * 6 + 2]}, V[3] = {rv[i * 6 + 3], rv[i * 6 + 4], rv[i * 6 + 5]};
    Elements el = {0, 0, 0, 0, 0, 0};
    const bool ok = orbital_elements(miu, R, V, el);
    out[i * 6] = el.a; out[i * 6 + 1] = el.e; out[i * 6 + 2] = el.i;
    out[i * 6 + 3] = el.omega; out[i * 6 + 4] = el.Omega; out[i * 6 + 5] = el.f;
    kind[i] = ok ? 6 : 0;
}

// calculate_state_information (satellite_function.py:257-315), six-element form
__global__ void state_info_kernel(const double* __restrict__ el, int64_t n, double miu, double* __restrict__ rv) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const double a = el[idx * 6], e = el[idx * 6 + 1], i = el[idx * 6 + 2], omega = el[idx * 6 + 3],
                 Omega = el[idx * 6 + 4], f = el[idx * 6 + 5];
    const double p = fabs(a * (1.0 - e * e));                 // :285
    const double u = omega + f;                               // :286
    double sO, cO, su, cu, si, ci, so, co;
    sincos(Omega, &sO, &cO); sincos(u, &su, &cu); sincos(i, &si, &ci); sincos(omega, &so, &co);
    const double k = p / (1.0 + e * cos(f));                  // :303
    rv[idx * 6 + 0] = k * (cO * cu - sO * su * ci);
    rv[idx * 6 + 1] = k * (sO * cu + cO * su * ci);
    rv[idx * 6 + 2] = k * (si * su);
    const double s = sqrt(miu / p);                           // :309
    rv[idx * 6 + 3] = s * (-cO * (su + e * so) - sO * (cu + e * co) * ci);
    rv[idx * 6 + 4] = s * (-sO * (su + e * so) + cO * (cu + e * co) * ci);
    rv[idx * 6 + 5] = s * (si * (cu + e * co));
}

// calculate_orbital_elements on every branch: the reference's list, zero-padded to 6 columns, and its length as the kind
__global__ void elements_all_kernel(const double* __restrict__ rv, int64_t n, double miu, double* __restrict__ out,
                                    int32_t* __restrict__ kind) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double R[3] = {rv[i * 6], rv[i * 6 + 1], rv[i * 6 + 2]}, V[3] = {rv[i * 6 + 3], rv[i * 6 + 4], rv[i * 6 + 5]};
    Elements el = {0, 0, 0, 0, 0, 0};
    kind[i] = orbital_elements<true, true>(miu, R, V, el);
    out[i * 6] = el.a; out[i * 6 + 1] = el.e; out[i * 6 + 2] = el.i;
    out[i * 6 + 3] = el.omega; out[i * 6 + 4] = el.Omega; out[i * 6 + 5] = el.f;
}

// calculate_state_information (satellite_function.py:287-315), the forms the parabolic and circular branches return:
//   NEL = 5: [p, i, omega, Omega, f], e = 1;   NEL = 4: [a, i, u, Omega], e = 0, p = a, omega = 0, f = u.
// Both run the six-element form's tail (:303-315) with the host libm's sin, cos and pow (glibm.cuh), so they are
// bit-identical to the reference's arithmetic.
template <int NEL>
__global__ void state_info_form_kernel(const double* __restrict__ el, int64_t n, double miu, double* __restrict__ rv) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const double* d = el + idx * NEL;
    double p, e, i, omega, Omega, f, u;
    if constexpr (NEL == 5) { p = d[0]; i = d[1]; omega = d[2]; Omega = d[3]; f = d[4]; e = 1.0; u = omega + f; }
    else { p = d[0]; i = d[1]; u = d[2]; Omega = d[3]; e = 0.0; omega = 0.0; f = u; }
    const double2 scO = glibm::call::sincos(Omega), scu = glibm::call::sincos(u), sci = glibm::call::sincos(i);
    const double2 sco = (NEL == 5) ? glibm::call::sincos(omega) : make_double2(0.0, 1.0);
    const double cf = (NEL == 5) ? glibm::call::cos(f) : scu.y;
    const double sO = scO.x, cO = scO.y, su = scu.x, cu = scu.y, si = sci.x, ci = sci.y, so = sco.x, co = sco.y;
    const double k = p / (1.0 + e * cf);                                  // :303
    rv[idx * 6 + 0] = k * (cO * cu - sO * su * ci);
    rv[idx * 6 + 1] = k * (sO * cu + cO * su * ci);
    rv[idx * 6 + 2] = k * (si * su);
    const double s = glibm::call::pow_half(miu / p);                     // :309
    rv[idx * 6 + 3] = s * (-cO * (su + e * so) - sO * (cu + e * co) * ci);
    rv[idx * 6 + 4] = s * (-sO * (su + e * so) + cO * (cu + e * co) * ci);
    rv[idx * 6 + 5] = s * (si * (cu + e * co));
}

// packed FFMA2 (fma.rn.f32x2) chain: the fp32 issue-rate ceiling of sm_100
__global__ void peak_ffma2_kernel(float* sink, int iters) {
    float2 a[8];
    const float2 m = make_float2(1.0000001f, 0.9999999f), c = make_float2(1e-7f, -1e-7f);
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = make_float2((threadIdx.x + k) * 1e-3f, (threadIdx.x + k) * 2e-3f);
#pragma unroll 16
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) a[k] = __ffma2_rn(a[k], m, c);
    }
    float s = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += a[k].x + a[k].y;
    if (s == -1.2345f) sink[0] = s;
}

inline int launch_status() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? SAT_OK : (int)e;
}
}  // namespace

extern "C" {

int sat_rk4_propagate(double* x, int64_t n, int64_t ld, double h, int substeps,
                      double mu, double re, double j2, void* stream) {
    if (!x) return SAT_ERR_NULL;
    if (n <= 0 || ld < n || substeps < 0) return SAT_ERR_SIZE;
    if ((ld & 1) || ((uintptr_t)x & 15)) return SAT_ERR_SIZE;
    if (substeps == 0) return SAT_OK;
    cudaStream_t s = (cudaStream_t)stream;
    // two states per thread only when that still leaves >= 4 warps per SM sub-partition in flight
    const bool ilp2 = n >= (int64_t)148 * 4 * 4 * 32 * 2;
    const int64_t threads_needed = ilp2 ? (n + 1) / 2 : n;
    const unsigned blocks = (unsigned)((threads_needed + kThreads - 1) / kThreads);
    if (j2 != 0.0) {
        if (ilp2) rk4_kernel<true, 2><<<blocks, kThreads, 0, s>>>(x, n, ld, substeps, h, mu, re, j2);
        else rk4_kernel<true, 1><<<blocks, kThreads, 0, s>>>(x, n, ld, substeps, h, mu, re, j2);
    } else {
        if (ilp2) rk4_kernel<false, 2><<<blocks, kThreads, 0, s>>>(x, n, ld, substeps, h, mu, re, j2);
        else rk4_kernel<false, 1><<<blocks, kThreads, 0, s>>>(x, n, ld, substeps, h, mu, re, j2);
    }
    return launch_status();
}

int sat_rk4_propagate_host(double* x_host, int64_t n, double* d_scratch, int64_t ld, double h,
                           int substeps, double mu, double re, double j2, void* stream) {
    if (!x_host || !d_scratch) return SAT_ERR_NULL;
    if (n <= 0 || ld < n) return SAT_ERR_SIZE;
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t ce = cudaMemcpy2DAsync(d_scratch, ld * sizeof(double), x_host, n * sizeof(double),
                                       n * sizeof(double), 6, cudaMemcpyHostToDevice, s);
    if (ce != cudaSuccess) return (int)ce;
    int rc = sat_rk4_propagate(d_scratch, n, ld, h, substeps, mu, re, j2, stream);
    if (rc) return rc;
    ce = cudaMemcpy2DAsync(x_host, n * sizeof(double), d_scratch, ld * sizeof(double),
                           n * sizeof(double), 6, cudaMemcpyDeviceToHost, s);
    if (ce != cudaSuccess) return (int)ce;
    ce = cudaStreamSynchronize(s);
    return ce == cudaSuccess ? SAT_OK : (int)ce;
}

int sat_state_eq(const double* x, double* f, int64_t n, int64_t ld, double mu, double re, double j2, void* stream) {
    if (!x || !f) return SAT_ERR_NULL;
    if (n <= 0 || ld < n) return SAT_ERR_SIZE;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    if (j2 != 0.0) state_eq_kernel<true><<<blocks, 128, 0, (cudaStream_t)stream>>>(x, f, n, ld, mu, re, j2);
    else state_eq_kernel<false><<<blocks, 128, 0, (cudaStream_t)stream>>>(x, f, n, ld, mu, re, j2);
    return launch_status();
}

int sat_cw_propagate(double* x, int64_t n, int64_t ld, const double* stm_host, void* stream) {
    if (!x || !stm_host) return SAT_ERR_NULL;
    if (n <= 0 || ld < n) return SAT_ERR_SIZE;
    Stm36 M;
    for (int k = 0; k < 36; ++k) M.m[k] = stm_host[k];
    cw_apply_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(x, n, ld, M);
    return launch_status();
}

int sat_orbital_elements(const double* rv, int64_t n, double miu, double* elements_out, int32_t* kind_out, void* stream) {
    if (!rv || !elements_out || !kind_out) return SAT_ERR_NULL;
    if (n <= 0) return SAT_ERR_SIZE;
    elements_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(rv, n, miu, elements_out, kind_out);
    return launch_status();
}

int sat_state_from_elements(const double* elements, int64_t n, double miu, double* rv_out, void* stream) {
    if (!elements || !rv_out) return SAT_ERR_NULL;
    if (n <= 0) return SAT_ERR_SIZE;
    state_info_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(elements, n, miu, rv_out);
    return launch_status();
}

int sat_orbital_elements_all(const double* rv, int64_t n, double miu, double* elements_out, int32_t* kind_out,
                             void* stream) {
    if (!rv || !elements_out || !kind_out) return SAT_ERR_NULL;
    if (n <= 0) return SAT_ERR_SIZE;
    elements_all_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(rv, n, miu, elements_out, kind_out);
    return launch_status();
}

int sat_state_from_elements_n(const double* elements, int64_t n, int n_el, double miu, double* rv_out, void* stream) {
    if (n_el == 6) return sat_state_from_elements(elements, n, miu, rv_out, stream);
    if (!elements || !rv_out) return SAT_ERR_NULL;
    if (n <= 0 || (n_el != 5 && n_el != 4)) return SAT_ERR_SIZE;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    if (n_el == 5) state_info_form_kernel<5><<<blocks, 128, 0, (cudaStream_t)stream>>>(elements, n, miu, rv_out);
    else state_info_form_kernel<4><<<blocks, 128, 0, (cudaStream_t)stream>>>(elements, n, miu, rv_out);
    return launch_status();
}

int sat_peak_fp64(double* sink, int blocks, int threads, int iters, double* flops_out_host, void* stream) {
    if (!sink) return SAT_ERR_NULL;
    if (blocks <= 0 || threads <= 0 || threads > 1024 || iters <= 0) return SAT_ERR_SIZE;
    peak_kernel<double><<<blocks, threads, 0, (cudaStream_t)stream>>>(sink, iters);
    if (flops_out_host) *flops_out_host = 2.0 * 16.0 * (double)iters * (double)blocks * (double)threads;
    return launch_status();
}

int sat_peak_fp32(float* sink, int blocks, int threads, int iters, double* flops_out_host, void* stream) {
    if (!sink) return SAT_ERR_NULL;
    if (blocks <= 0 || threads <= 0 || threads > 1024 || iters == 0) return SAT_ERR_SIZE;
    // 16 FMAs per thread per iteration either way: 16 scalar FFMA chains, or (iters < 0) 8 packed FFMA2 chains
    if (iters < 0) { iters = -iters; peak_ffma2_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(sink, iters); }
    else peak_kernel<float><<<blocks, threads, 0, (cudaStream_t)stream>>>(sink, iters);
    if (flops_out_host) *flops_out_host = 2.0 * 16.0 * (double)iters * (double)blocks * (double)threads;
    return launch_status();
}

}  // extern "C"
