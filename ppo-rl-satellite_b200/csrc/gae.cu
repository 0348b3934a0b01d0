// gae.cu -- K4: GAE reverse scan + advantage normalisation for sm_100a.
//
// Reference behaviour replaced: ppo_continuous.py:198-210.
//   deltas = r + gamma*(1-dw)*vs_ - vs                    (torch fp32, separate ops)
//   gae    = delta + gamma*lamda*gae*(1-d)                (numpy float32 scalars under numpy 2)
//   v_target = adv + vs;  adv = (adv - mean)/(std_unbiased + 1e-5)
// The recursion is reproduced with explicit round-to-nearest fp32 ops in the reference's order,
// so advantages are bit-identical to the reference (bar: 1e-6).
//
// Layouts: time-major [T][N] (one thread per env walks t = T-1..0, every access coalesced, v[t+1]
// carried in a register), and the reference's flat (B,1) buffer of a single env, which is staged
// through shared memory in chunks and scanned there.
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/satb200.h"

namespace {

__device__ __forceinline__ float gae_delta(float r, float gamma, float dw, float vnext, float v) {
    // (r + ((gamma * (1 - dw)) * vs_)) - vs
    return __fsub_rn(__fadd_rn(r, __fmul_rn(__fmul_rn(gamma, __fsub_rn(1.0f, dw)), vnext)), v);
}
__device__ __forceinline__ float gae_step(float delta, float gl, float gae, float d) {
    // delta + ((gl * gae) * (1 - d))
    return __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, gae), __fsub_rn(1.0f, d)));
}

// Time-major GAE, tiled: a CTA owns 32 adjacent envs (one 128-byte row segment per time step) and walks time in tiles of
// kGaeTile steps from the end of the rollout. All 8 warps stream a tile in (r, v, done -> registers while the previous tile
// is being scanned), stage it in shared memory and turn it into deltas; warp 0 then runs the strictly sequential recursion
// for its 32 envs out of shared memory (3 dependent fp32 operations per step, rounded exactly like the reference's numpy
// float32 scalars), and all warps write adv / v_target back with full-line stores. The loads of tile i-1 are in flight during
// the scan of tile i, so the kernel is limited by HBM (17 B/sample), not by the length of one env's dependency chain -
// the one-thread-per-env form reached 7 % of HBM at the config-5 shard (T = 2048, N = 8192: 64 CTAs, 2048 dependent steps).
constexpr int kGaeTile = 64;      // time steps per tile
// envs per CTA (template parameter): 32 (a 128-byte row segment) when there are enough envs to fill the GPU with such CTAs; at
// the config-5 shard (N = 8192) that gives only 256 CTAs = 1.7 per SM, each a serial chain of 32 tiles, and the kernel sat at
// 0.37 of HBM, so narrower CTAs (16 or 8 envs: 64- / 32-byte segments, still whole sectors) are used to put more independent
// scans on every SM.
constexpr int kGaeThreads = 256;

template <int kGaeEnvs>
__global__ void __launch_bounds__(kGaeThreads)
gae_time_major_kernel(const float* __restrict__ r, const float* __restrict__ v, const uint8_t* __restrict__ done,
                      const float* __restrict__ r_scale, int64_t T, int64_t N, float gamma, float gl,
                      float* __restrict__ adv, float* __restrict__ vt) {
    constexpr int kGaePer = kGaeTile * kGaeEnvs / kGaeThreads;   // elements per thread per tile
    __shared__ float s_x[kGaeTile][kGaeEnvs];      // reward, then delta, then gae
    __shared__ float s_v[kGaeTile][kGaeEnvs];      // vs
    __shared__ float s_d[kGaeTile][kGaeEnvs];      // done as 0 / 1
    __shared__ float s_vtop[kGaeEnvs];             // v of the row above the tile (t + 1 of its last step)
    __shared__ float s_gae[kGaeEnvs];              // recursion carry
    const int lane_e = threadIdx.x & (kGaeEnvs - 1);
    const int row0 = threadIdx.x / kGaeEnvs;       // 0..7: the thread handles rows row0, row0 + 8, ...
    const int64_t e = (int64_t)blockIdx.x * kGaeEnvs + lane_e;
    const bool ev = e < N;
    if (threadIdx.x < kGaeEnvs) { s_gae[threadIdx.x] = 0.0f; s_vtop[threadIdx.x] = ev ? v[T * N + e] : 0.0f; }
    // prefetch registers hold the RAW loaded values: any arithmetic on them here would wait for each load in turn and
    // serialise the tile's 24 loads per thread into 8 DRAM round trips (measured: 7 us per tile instead of < 1)
    float pr[kGaePer], pv[kGaePer];
    uint8_t pd[kGaePer];
    // tiles cover [lo, lo + len), processed from the end of the rollout; the first (topmost) tile may be partial
    int64_t hi = T;
    int64_t lo = ((T - 1) / kGaeTile) * kGaeTile;
    auto prefetch = [&](int64_t lo_, int len_) {
#pragma unroll
        for (int k = 0; k < kGaePer; ++k) {
            const int row = row0 + k * (kGaeThreads / kGaeEnvs);
            if (row < len_ && ev) {
                const int64_t i = (lo_ + row) * N + e;
                pr[k] = r[i]; pv[k] = v[i]; pd[k] = done[i];
            } else { pr[k] = 0.0f; pv[k] = 0.0f; pd[k] = 0; }
        }
    };
    prefetch(lo, (int)(hi - lo));
    while (hi > 0) {
        const int len = (int)(hi - lo);
        __syncthreads();                            // previous tile fully written out; s_vtop / s_gae visible
#pragma unroll
        for (int k = 0; k < kGaePer; ++k) {
            const int row = row0 + k * (kGaeThreads / kGaeEnvs);
            float rr = pr[k];
            if (r_scale && row < len) rr = __fmul_rn(rr, r_scale[lo + row]);
            s_x[row][lane_e] = rr; s_v[row][lane_e] = pv[k]; s_d[row][lane_e] = pd[k] ? 1.0f : 0.0f;
        }
        const int64_t nlo = lo - kGaeTile;
        if (lo > 0) prefetch(nlo, kGaeTile);        // next tile's loads fly during the delta pass and the scan
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kGaePer; ++k) {
            const int row = row0 + k * (kGaeThreads / kGaeEnvs);
            // besides the delta, the pass leaves the recursion coefficient c = gl (1 - d) in s_d: (gl gae)(1 - d) with
            // (1 - d) in {0, 1} has the bits of (gl (1 - d)) gae (a product with 1 is exact, one with 0 is a zero of the same
            // sign), so the scan's dependent chain is one multiply and one add per step instead of two multiplies, a
            // subtraction and an add. Rows past a partial top tile get delta = c = 0: the scan then always runs kGaeTile steps
            // (ncu: 59 % of the kernel's warp time was the other warps waiting for a 28-instruction-per-step scan loop)
            float dl = 0.0f, c = 0.0f;
            if (row < len) {
                const float d = s_d[row][lane_e];
                const float vnext = (row == len - 1) ? s_vtop[lane_e] : s_v[row + 1][lane_e];
                dl = gae_delta(s_x[row][lane_e], gamma, d, vnext, s_v[row][lane_e]);
                c = __fmul_rn(gl, __fsub_rn(1.0f, d));
            }
            s_x[row][lane_e] = dl; s_d[row][lane_e] = c;
        }
        __syncthreads();
        if (threadIdx.x < kGaeEnvs) {
            float gae = s_gae[lane_e];
#pragma unroll 16
            for (int row = kGaeTile - 1; row >= 0; --row) {
                gae = __fadd_rn(s_x[row][lane_e], __fmul_rn(s_d[row][lane_e], gae));      // delta + (gl (1 - d)) gae
                s_x[row][lane_e] = gae;
            }
            s_gae[lane_e] = gae;
        }
        __syncthreads();
        if (ev) {
#pragma unroll
            for (int k = 0; k < kGaePer; ++k) {
                const int row = row0 + k * (kGaeThreads / kGaeEnvs);
                if (row < len) {
                    const int64_t i = (lo + row) * N + e;
                    const float g = s_x[row][lane_e];
                    adv[i] = g;
                    vt[i] = __fadd_rn(g, s_v[row][lane_e]);                  // :208
                }
            }
        }
        if (threadIdx.x < kGaeEnvs) s_vtop[lane_e] = s_v[0][lane_e];         // v[lo] is v(t + 1) for the tile below
        hi = lo; lo = nlo;
    }
}

constexpr int kFlatChunk = 4096;

__global__ void __launch_bounds__(256)
gae_flat_kernel(const float* __restrict__ r, const float* __restrict__ vs, const float* __restrict__ vs_next,
                const float* __restrict__ dw, const float* __restrict__ done, int64_t B, float gamma, float gl,
                float* __restrict__ adv, float* __restrict__ vt) {
    // single CTA: chunks of the buffer are staged into shared memory (delta, 1-d), scanned in reverse by
    // one thread (the recurrence is strictly sequential and must round like the reference), then the
    // chunk's advantages are written back cooperatively.
    __shared__ float s_delta[kFlatChunk];
    __shared__ float s_keep[kFlatChunk];
    __shared__ float s_carry;
    if (threadIdx.x == 0) s_carry = 0.0f;
    __syncthreads();
    for (int64_t hi = B; hi > 0; hi -= kFlatChunk) {
        const int64_t lo = hi > kFlatChunk ? hi - kFlatChunk : 0;
        const int len = (int)(hi - lo);
        for (int j = threadIdx.x; j < len; j += blockDim.x) {
            const int64_t i = lo + j;
            s_delta[j] = gae_delta(r[i], gamma, dw[i], vs_next[i], vs[i]);
            s_keep[j] = done[i];
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            float gae = s_carry;
            for (int j = len - 1; j >= 0; --j) {
                gae = gae_step(s_delta[j], gl, gae, s_keep[j]);
                s_delta[j] = gae;
            }
            s_carry = gae;
        }
        __syncthreads();
        for (int j = threadIdx.x; j < len; j += blockDim.x) {
            const int64_t i = lo + j;
            const float g = s_delta[j];
            adv[i] = g;
            vt[i] = __fadd_rn(g, vs[i]);
        }
        __syncthreads();
    }
}

constexpr int kMomThreads = 256;

__global__ void __launch_bounds__(kMomThreads)
moments_partial_kernel(const float* __restrict__ x, int64_t count, double* __restrict__ partial) {
    __shared__ double s_sum[kMomThreads / 32], s_sq[kMomThreads / 32];
    double sum = 0.0, sq = 0.0;
    // four independent 128-bit loads in flight per thread; per-thread accumulation order is fixed -> deterministic
    const int64_t stride = (int64_t)gridDim.x * kMomThreads;
    const int64_t tid = (int64_t)blockIdx.x * kMomThreads + threadIdx.x;
    if ((reinterpret_cast<uintptr_t>(x) & 15) == 0) {
        const float4* x4 = reinterpret_cast<const float4*>(x);
        const int64_t n4 = count >> 2;
        for (int64_t i = tid; i < n4; i += 4 * stride) {
            float4 q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) q[u] = (i + u * stride < n4) ? x4[i + u * stride] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const double a = q[u].x, b = q[u].y, c = q[u].z, d = q[u].w;
                sum += (a + b) + (c + d); sq += (a * a + b * b) + (c * c + d * d);
            }
        }
        for (int64_t i = (n4 << 2) + tid; i < count; i += stride) { const double v = (double)x[i]; sum += v; sq += v * v; }
    } else {
        for (int64_t i = tid; i < count; i += stride) { const double v = (double)x[i]; sum += v; sq += v * v; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, off);
        sq += __shfl_xor_sync(0xffffffffu, sq, off);
    }
    if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = sum; s_sq[threadIdx.x >> 5] = sq; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < kMomThreads / 32; ++w) { a += s_sum[w]; b += s_sq[w]; }
        partial[2 * blockIdx.x] = a; partial[2 * blockIdx.x + 1] = b;
    }
}

__global__ void __launch_bounds__(256)
moments_final_kernel(const double* __restrict__ partial, int nblocks, int64_t count, double* __restrict__ sums) {
    // fixed summation order (thread-strided, then a fixed tree): bitwise reproducible from run to run
    __shared__ double s_a[256], s_b[256];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += 256) { a += partial[2 * i]; b += partial[2 * i + 1]; }
    s_a[threadIdx.x] = a; s_b[threadIdx.x] = b;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) { s_a[threadIdx.x] += s_a[threadIdx.x + off]; s_b[threadIdx.x] += s_b[threadIdx.x + off]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { sums[0] = s_a[0]; sums[1] = s_b[0]; sums[2] = (double)count; }
}

__global__ void __launch_bounds__(256)
adv_normalize_kernel(float* __restrict__ adv, int64_t count, const double* __restrict__ sums) {
    const double n = sums[2];
    const double mean = sums[0] / n;
    double var = (sums[1] - n * mean * mean) / (n - 1.0);      // torch.std(): unbiased
    if (var < 0.0) var = 0.0;
    const float m = (float)mean, den = __fadd_rn((float)sqrt(var), 1e-5f);
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    if ((reinterpret_cast<uintptr_t>(adv) & 15) == 0) {
        float4* a4 = reinterpret_cast<float4*>(adv);
        const int64_t n4 = count >> 2;
        for (int64_t i = tid; i < n4; i += stride) {
            float4 q = a4[i];
            q.x = __fdiv_rn(__fsub_rn(q.x, m), den); q.y = __fdiv_rn(__fsub_rn(q.y, m), den);       // ppo_continuous.py:210
            q.z = __fdiv_rn(__fsub_rn(q.z, m), den); q.w = __fdiv_rn(__fsub_rn(q.w, m), den);
            a4[i] = q;
        }
        for (int64_t i = (n4 << 2) + tid; i < count; i += stride) adv[i] = __fdiv_rn(__fsub_rn(adv[i], m), den);
    } else {
        for (int64_t i = tid; i < count; i += stride) adv[i] = __fdiv_rn(__fsub_rn(adv[i], m), den);
    }
}

inline int launch_status() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? SAT_OK : (int)e;
}
constexpr int kMomBlocks = 148 * 8;   // 8 per SM

}  // namespace

extern "C" {

int sat_gae(const float* r, const float* v, const uint8_t* done, const float* r_scale, int64_t T, int64_t N,
            double gamma, double lamda, float* adv, float* v_target, void* stream) {
    if (!r || !v || !done || !adv || !v_target) return SAT_ERR_NULL;
    if (T <= 0 || N <= 0) return SAT_ERR_SIZE;
    // :205 multiplies the python floats first and weak-casts the double product to fp32; :203 multiplies an fp32 tensor
    // by gamma, which torch rounds to fp32 first
    const float gl = (float)(gamma * lamda), g32 = (float)gamma;
    // at least ~6 CTAs per SM (148 SMs) where the env count allows it
    if (N >= 32 * 888) gae_time_major_kernel<32><<<(unsigned)((N + 31) / 32), kGaeThreads, 0, (cudaStream_t)stream>>>(r, v, done, r_scale, T, N, g32, gl, adv, v_target);
    else if (N >= 16 * 296) gae_time_major_kernel<16><<<(unsigned)((N + 15) / 16), kGaeThreads, 0, (cudaStream_t)stream>>>(r, v, done, r_scale, T, N, g32, gl, adv, v_target);
    else gae_time_major_kernel<8><<<(unsigned)((N + 7) / 8), kGaeThreads, 0, (cudaStream_t)stream>>>(r, v, done, r_scale, T, N, g32, gl, adv, v_target);
    return launch_status();
}

int sat_gae_flat(const float* r, const float* vs, const float* vs_next, const float* dw, const float* done,
                 int64_t B, double gamma, double lamda, float* adv, float* v_target, void* stream) {
    if (!r || !vs || !vs_next || !dw || !done || !adv || !v_target) return SAT_ERR_NULL;
    if (B <= 0) return SAT_ERR_SIZE;
    const float gl = (float)(gamma * lamda), g32 = (float)gamma;          // as in sat_gae
    gae_flat_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(r, vs, vs_next, dw, done, B, g32, gl, adv, v_target);
    return launch_status();
}

int sat_adv_moments(const float* adv, int64_t count, double* sums, void* workspace, void* stream) {
    if (!adv || !sums || !workspace) return SAT_ERR_NULL;
    if (count <= 0) return SAT_ERR_SIZE;
    cudaStream_t s = (cudaStream_t)stream;
    int nblocks = (int)((count + kMomThreads - 1) / kMomThreads);
    if (nblocks > kMomBlocks) nblocks = kMomBlocks;
    moments_partial_kernel<<<nblocks, kMomThreads, 0, s>>>(adv, count, (double*)workspace);
    int rc = launch_status();
    if (rc) return rc;
    moments_final_kernel<<<1, 256, 0, s>>>((const double*)workspace, nblocks, count, sums);
    return launch_status();
}

int sat_adv_normalize(float* adv, int64_t count, const double* sums, void* stream) {
    if (!adv || !sums) return SAT_ERR_NULL;
    if (count <= 0) return SAT_ERR_SIZE;
    int64_t nb = (count / 4 + 255) / 256;
    if (nb < 1) nb = 1;
    if (nb > 148 * 16) nb = 148 * 16;
    adv_normalize_kernel<<<(unsigned)nb, 256, 0, (cudaStream_t)stream>>>(adv, count, sums);
    return launch_status();
}

}  // extern "C"
