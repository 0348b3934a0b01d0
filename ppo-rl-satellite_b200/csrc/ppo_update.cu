// ppo_update.cu -- fused PPO minibatch step for the 18-256-256-{3,1} MLPs (SURVEY.md s8 f.1) on sm_100a.
//
// Reference behaviour replaced: the body of the K-epoch loop of PPO_continuous.update (ppo_continuous.py:216-239):
//     dist_now = actor.get_dist(s[index]); ratios = exp(sum logp_now - sum logp_old)
//     actor_loss = -min(ratios*adv, clamp(ratios, 1-eps, 1+eps)*adv) - entropy_coef*entropy;  .mean().backward()
//     critic_loss = mse_loss(v_target[index], critic(s[index]));                             .backward()
//     clip_grad_norm_(0.5); Adam(eps=1e-5).step()                                             (:161-163, 228-238)
// fp32 CUDA-core FFMA2 (the reference trains in fp32 and the north star rules tensor cores out).
//
// Per network and minibatch, five launches:
//   ppo_fb_kernel     one CTA per 64 rows, the same 64 x 256 register-tile GEMM as the actor kernel, three times:
//                     h1 = act(W1 x), h2 = act(W2 h1) (W2^T streamed by TMA bulk copies), heads + loss gradient per row,
//                     dz2 = (dz3 W3) act'(h2), dh1 = dz2 W2 (fc2.weight streamed in its torch layout), dz1 = dh1 act'(h1).
//                     h1 / dz2 / dz1 go to HBM once for the weight gradients; dW3, db2, db3, dlog_std and the loss are
//                     reduced per CTA.
//   ppo_wgrad2_kernel dW2 = dz2^T h1, split-K over 74 row slabs x 4 column blocks (296 CTAs = 2 per SM), both operands
//                     streamed k-major through a 4-stage TMA pipeline.
//   ppo_wgrad1_kernel dW1 = dz1^T x and db1, a streaming pass over dz1 (3-stage TMA pipeline).
//   colsum_kernel     deterministic sum of the per-CTA / per-slab partials into the flat gradient.
//   ppo_adam_kernel   one 8-CTA cluster: gradient norm through distributed shared memory, clip, Adam, and the packed
//                     (transposed) weight image for the next forward.
// The *_stats entry points run the STATS instantiations of the forward/backward and Adam kernels: the actor's row threads also
// reduce the per-row diagnostics (surrogate, entropy, approximate KL, clipped) into part_stat, one more colsum launch writes them
// to grads[n + 2 .. n + 6) (so the gradient exchange carries them), and the Adam kernel adds the global minibatch means, the
// gradient norm and the clip coefficient to a caller-owned fp64 record. Gradients and parameters are bit-identical to the
// default kernels'.
#include <cooperative_groups.h>
#include "mlp_tile.cuh"
#include "ppo_fb_tc.cuh"
#include <cstdlib>

namespace cg = cooperative_groups;

namespace {
using namespace mlp;

constexpr int W2_SLABS = 74;          // 4 column blocks x 74 slabs = 296 CTAs
constexpr int W1_SLABS = 592;
constexpr int WG_STAGES = 4;
constexpr int XS_LD = 32;             // gathered observation rows, padded to 32 floats

__host__ __device__ inline int off_b3(int heads) { return SAT_PPO_OFF_W3 + heads * HID; }
__host__ __device__ inline int param_floats(int heads) { return SAT_PPO_PARAM_FLOATS(heads); }

struct Workspace {
    float *h1, *dz2b, *dz1, *xs, *part_head, *part_scal, *part_w2, *part_w1, *part_b1, *part_stat;
    unsigned char* tc_image;         // the tensor-core forward/backward kernel's split, swizzled weight operands
    int64_t mp, tiles;
};
constexpr int64_t MP_ALIGN = 128;    // rows are padded to the tensor-core kernel's 128-row tile (two 64-row FFMA tiles)
__host__ inline int64_t ws_floats(int64_t mb) {
    const int64_t mp = (mb + MP_ALIGN - 1) / MP_ALIGN * MP_ALIGN, tiles = mp / M;
    return mp * HID * 3 + mp * XS_LD + tiles * 4 * HID + tiles * 8 + (int64_t)W2_SLABS * HID * HID +
           (int64_t)W1_SLABS * (HID * IN + HID) + SAT_PPO_TC_IMAGE_BYTES / 4 + 64 + tiles * 8;
}
__host__ inline Workspace ws_carve(float* base, int64_t mb) {
    Workspace w;
    w.mp = (mb + MP_ALIGN - 1) / MP_ALIGN * MP_ALIGN; w.tiles = w.mp / M;
    float* p = base;
    w.h1 = p; p += w.mp * HID;
    w.dz2b = p; p += w.mp * HID;
    w.dz1 = p; p += w.mp * HID;
    w.xs = p; p += w.mp * XS_LD;
    w.part_head = p; p += w.tiles * 4 * HID;
    w.part_scal = p; p += w.tiles * 8;
    w.part_w2 = p; p += (int64_t)W2_SLABS * HID * HID;
    w.part_w1 = p; p += (int64_t)W1_SLABS * HID * IN;
    w.part_b1 = p; p += (int64_t)W1_SLABS * HID;
    w.tc_image = reinterpret_cast<unsigned char*>(p + ((64 - ((p - base) & 63)) & 63));     // 256-byte aligned (base is 16-byte aligned)
    w.part_stat = base + ws_floats(mb) - w.tiles * 8;                                        // [tiles][8], the last region
    return w;
}

struct __align__(128) FbSmem {
    float hT[HID * H1_LD];           // h1^T during the forward, dz2^T during the backward
    float wt[NSTAGE][KT * HID];      // weight k-tiles; W1^T and the reduction scratch alias this region
    float xT[IN * M];
    float w3[ACTP * HID];
    float pre[M * ACTP];
    float dz3[M * ACTP];
    float red[2][8];
    uint64_t full[NSTAGE];
    uint64_t bar_misc;
};
static_assert(NWARPS * 4 * HID * 4 <= NSTAGE * KT * HID * 4, "reduction scratch must fit in the stage region");
struct __align__(128) FbSmemStats : FbSmem {
    float stat[2][4];                // per-warp partial sums of the diagnostics (STATS instantiation)
};

__device__ __forceinline__ float act_grad(float h, int use_tanh) { return use_tanh ? 1.0f - h * h : (h > 0.0f ? 1.0f : 0.0f); }
__device__ __forceinline__ float& acc_ref(float2 (&acc)[RT][NP], int i, int c, int q) {
    float2& v = acc[i][c * 2 + (q >> 1)];
    return (q & 1) ? v.y : v.x;
}
__device__ __forceinline__ void acc_zero(float2 (&acc)[RT][NP]) {
#pragma unroll
    for (int i = 0; i < RT; ++i)
#pragma unroll
        for (int j = 0; j < NP; ++j) acc[i][j] = make_float2(0.0f, 0.0f);
}

// STATS (actor only): the row threads also reduce the per-row diagnostics (surrogate, entropy, approximate KL, clipped), each
// scaled by inv_n like the loss, into part_stat [tile][8] (the first four entries)
template <bool CRITIC, bool STATS>
__global__ void __launch_bounds__(THREADS, 2)
ppo_fb_kernel(const float* __restrict__ packed, const float* __restrict__ w2, int use_tanh, float max_action,
              const float* __restrict__ s, const float* __restrict__ a, const float* __restrict__ old_logp,
              const float* __restrict__ adv, const float* __restrict__ v_target, const int64_t* __restrict__ index,
              int64_t n, float inv_n, float epsilon, float entropy_coef,
              float* __restrict__ h1g, float* __restrict__ dz2b, float* __restrict__ dz1g, float* __restrict__ xs,
              float* __restrict__ part_head, float* __restrict__ part_scal, int64_t mp, float* __restrict__ part_stat) {
    static_assert(!(STATS && CRITIC), "the critic has no per-row diagnostics beyond its loss");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    FbSmem& sm = *reinterpret_cast<FbSmem*>(smem_raw);
    const int tid = threadIdx.x, tx = tid % TXN, ty = tid / TXN, warp = tid >> 5;
    const int64_t row0 = (int64_t)blockIdx.x * M;
    constexpr int heads = CRITIC ? 1 : 3;

    if (tid == 0) {
        mbar_init(&sm.full[0], 1); mbar_init(&sm.full[1], 1); mbar_init(&sm.bar_misc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(&sm.bar_misc, IN * HID * 4 + ACTP * HID * 4);
        bulk_g2s(&sm.wt[0][0], packed + OFF_W1T, IN * HID * 4, &sm.bar_misc);
        bulk_g2s(&sm.w3[0], packed + OFF_W3, ACTP * HID * 4, &sm.bar_misc);
    }

    // ---------------- gather the minibatch rows (ppo_continuous.py:217 s[index]) -> xT, and the padded copy for dW1
    for (int idx = tid; idx < M * IN; idx += THREADS) {
        const int row = idx / IN, d = idx - row * IN;
        const int64_t g = row0 + row;
        float v = 0.0f;
        if (g < n) { const int64_t src = index ? index[g] : g; v = s[src * IN + d]; }
        sm.xT[d * M + row] = v;
    }
    __syncthreads();
    for (int idx = tid; idx < M * XS_LD; idx += THREADS) {
        const int row = idx / XS_LD, d = idx - row * XS_LD;
        xs[(row0 + row) * XS_LD + d] = d < IN ? sm.xT[d * M + row] : 0.0f;
    }

    // ---------------- layer 1
    float2 acc[RT][NP];
    acc_zero(acc);
    mbar_wait(&sm.bar_misc, 0);
    tile_fma<IN>(acc, sm.xT, M, &sm.wt[0][0], ty, tx);
#pragma unroll
    for (int c = 0; c < NC; ++c)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = c * CSTR + tx * 4 + q;
            const float bias = __ldg(packed + OFF_B1 + j);
#pragma unroll
            for (int i = 0; i < RT; ++i) acc_ref(acc, i, c, q) = activate(acc_ref(acc, i, c, q) + bias, use_tanh);
#pragma unroll
            for (int i4 = 0; i4 < RT / 4; ++i4) {
                float4 o;
                o.x = acc_ref(acc, i4 * 4 + 0, c, q); o.y = acc_ref(acc, i4 * 4 + 1, c, q);
                o.z = acc_ref(acc, i4 * 4 + 2, c, q); o.w = acc_ref(acc, i4 * 4 + 3, c, q);
                *reinterpret_cast<float4*>(&sm.hT[j * H1_LD + ty * RT + i4 * 4]) = o;
            }
        }
    // h1 to HBM, row-major [mp][256]: re-read by this same thread for dz1 and streamed by the dW2 kernel
#pragma unroll
    for (int i = 0; i < RT; ++i)
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const float2 lo = acc[i][c * 2], hi = acc[i][c * 2 + 1];
            *reinterpret_cast<float4*>(h1g + (row0 + ty * RT + i) * HID + c * CSTR + tx * 4) = make_float4(lo.x, lo.y, hi.x, hi.y);
        }
    __syncthreads();      // h1T complete; W1^T region free for the W2^T stages

    // ---------------- layer 2 forward: stream W2^T
    constexpr int NT = HID / KT;
    if (tid == 0) {
#pragma unroll
        for (int st = 0; st < NSTAGE; ++st) {
            mbar_expect_tx(&sm.full[st], KT * HID * 4);
            bulk_g2s(&sm.wt[st][0], packed + OFF_W2T + st * KT * HID, KT * HID * 4, &sm.full[st]);
        }
    }
    acc_zero(acc);
#pragma unroll 1
    for (int t = 0; t < NT; ++t) {
        const int st = t & 1;
        mbar_wait(&sm.full[st], (t >> 1) & 1);
        tile_fma<KT>(acc, sm.hT + t * KT * H1_LD, H1_LD, &sm.wt[st][0], ty, tx);
        __syncthreads();
        if (tid == 0 && t + NSTAGE < NT) {
            mbar_expect_tx(&sm.full[st], KT * HID * 4);
            bulk_g2s(&sm.wt[st][0], packed + OFF_W2T + (t + NSTAGE) * KT * HID, KT * HID * 4, &sm.full[st]);
        }
    }

    // ---------------- h2 in place, head pre-activations
    {
        float part[RT][heads];
#pragma unroll
        for (int i = 0; i < RT; ++i)
#pragma unroll
            for (int h = 0; h < heads; ++h) part[i][h] = 0.0f;
#pragma unroll
        for (int c = 0; c < NC; ++c)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int j = c * CSTR + tx * 4 + q;
                const float bias = __ldg(packed + OFF_B2 + j);
                float w[heads];
#pragma unroll
                for (int h = 0; h < heads; ++h) w[h] = sm.w3[h * HID + j];
#pragma unroll
                for (int i = 0; i < RT; ++i) {
                    const float hv = activate(acc_ref(acc, i, c, q) + bias, use_tanh);
                    acc_ref(acc, i, c, q) = hv;
#pragma unroll
                    for (int h = 0; h < heads; ++h) part[i][h] = fmaf(hv, w[h], part[i][h]);
                }
            }
#pragma unroll
        for (int off = 1; off < TXN; off <<= 1)
#pragma unroll
            for (int i = 0; i < RT; ++i)
#pragma unroll
                for (int h = 0; h < heads; ++h) part[i][h] += __shfl_xor_sync(0xffffffffu, part[i][h], off);
        if (tx == 0) {
#pragma unroll
            for (int i = 0; i < RT; ++i)
#pragma unroll
                for (int h = 0; h < heads; ++h) sm.pre[(ty * RT + i) * ACTP + h] = part[i][h];
        }
    }
    __syncthreads();

    // ---------------- per-row loss and its gradient w.r.t. the head pre-activations (first two warps, one row each)
    if (tid < M) {
        const int64_t g = row0 + tid;
        float d3[3] = {0.0f, 0.0f, 0.0f}, dls[3] = {0.0f, 0.0f, 0.0f}, loss = 0.0f;
        [[maybe_unused]] float stat[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        if (g < n) {
            const int64_t src = index ? index[g] : g;
            if (CRITIC) {
                const float v = sm.pre[tid * ACTP] + __ldg(packed + OFF_B3);
                const float diff = v - v_target[src];
                loss = diff * diff * inv_n;                                                    // :233
                d3[0] = 2.0f * diff * inv_n;
            } else {
                float mean[3], sd[3], x[3], th[3], lsum = 0.0f, ent = 0.0f;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    th[k] = tanhf(sm.pre[tid * ACTP + k] + __ldg(packed + OFF_B3 + k));
                    mean[k] = max_action * th[k];
                    const float ls = __ldg(packed + OFF_LS + k);
                    sd[k] = expf(ls);
                    x[k] = a[src * 3 + k];
                    const float diff = x[k] - mean[k];
                    lsum += -(diff * diff) / (2.0f * sd[k] * sd[k]) - ls - 0.9189385332046727f - old_logp[src * 3 + k];   // :219-221
                    ent += 1.4189385332046727f + ls;                                           // :218 Normal.entropy()
                }
                const float ratio = expf(lsum);
                const float A = adv[src];
                const float surr1 = ratio * A;
                const bool inside = ratio >= 1.0f - epsilon && ratio <= 1.0f + epsilon;
                const float surr2 = fminf(fmaxf(ratio, 1.0f - epsilon), 1.0f + epsilon) * A;   // :224
                loss = (-fminf(surr1, surr2) - entropy_coef * ent) * inv_n;                    // :225, .mean() :228
                // d(-min)/d ratio: torch.min splits the gradient on ties and clamp passes it only inside the range
                const float pass = surr1 < surr2 ? 1.0f : (surr1 == surr2 ? (inside ? 1.0f : 0.5f) : 0.0f);
                const float gs = -A * pass * ratio * inv_n;                                    // d loss / d (sum logp)
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float diff = x[k] - mean[k], iv = 1.0f / (sd[k] * sd[k]);
                    d3[k] = gs * diff * iv * max_action * (1.0f - th[k] * th[k]);
                    dls[k] = gs * (diff * diff * iv - 1.0f) - entropy_coef * inv_n;
                }
                if constexpr (STATS) {
                    // approximate KL (ratio - 1) - log ratio as expm1 - lsum: (expf(lsum) - 1) - lsum cancels in fp32
                    stat[0] = -fminf(surr1, surr2) * inv_n;
                    stat[1] = ent * inv_n;
                    stat[2] = (expm1f(lsum) - lsum) * inv_n;
                    stat[3] = fabsf(ratio - 1.0f) > epsilon ? inv_n : 0.0f;
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) sm.dz3[tid * ACTP + k] = d3[k];
        float red[8] = {d3[0], d3[1], d3[2], dls[0], dls[1], dls[2], loss, 0.0f};
        if (CRITIC) { red[1] = loss; red[6] = 0.0f; }
#pragma unroll
        for (int k = 0; k < 7; ++k)
#pragma unroll
            for (int off = 16; off; off >>= 1) red[k] += __shfl_xor_sync(0xffffffffu, red[k], off);
        if ((tid & 31) == 0)
#pragma unroll
            for (int k = 0; k < 8; ++k) sm.red[warp][k] = red[k];
        if constexpr (STATS) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
#pragma unroll
                for (int off = 16; off; off >>= 1) stat[k] += __shfl_xor_sync(0xffffffffu, stat[k], off);
            if ((tid & 31) == 0)
#pragma unroll
                for (int k = 0; k < 4; ++k) reinterpret_cast<FbSmemStats*>(smem_raw)->stat[warp][k] = stat[k];
        }
    }
    __syncthreads();
    if (tid < 8) part_scal[(int64_t)blockIdx.x * 8 + tid] = sm.red[0][tid] + sm.red[1][tid];
    if constexpr (STATS) {
        const FbSmemStats& sst = *reinterpret_cast<const FbSmemStats*>(smem_raw);
        if (tid >= 8 && tid < 12) part_stat[(int64_t)blockIdx.x * 8 + tid - 8] = sst.stat[0][tid - 8] + sst.stat[1][tid - 8];
    }

    // ---------------- dz2 = (dz3 W3) act'(h2) in place; per-CTA partial sums of dW3 (rows 0..heads-1) and db2 (row 3)
    {
        float d3[RT][heads];
#pragma unroll
        for (int i = 0; i < RT; ++i)
#pragma unroll
            for (int h = 0; h < heads; ++h) d3[i][h] = sm.dz3[(ty * RT + i) * ACTP + h];
        float* scratch = &sm.wt[0][0];                       // [NWARPS][4 rows][HID]
#pragma unroll
        for (int c = 0; c < NC; ++c)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int j = c * CSTR + tx * 4 + q;
                float w[heads], sw[heads], sb = 0.0f;
#pragma unroll
                for (int h = 0; h < heads; ++h) { w[h] = sm.w3[h * HID + j]; sw[h] = 0.0f; }
#pragma unroll
                for (int i = 0; i < RT; ++i) {
                    const float hv = acc_ref(acc, i, c, q);
                    float dh = 0.0f;
#pragma unroll
                    for (int h = 0; h < heads; ++h) { dh = fmaf(d3[i][h], w[h], dh); sw[h] = fmaf(hv, d3[i][h], sw[h]); }
                    const float dz = dh * act_grad(hv, use_tanh);
                    sb += dz;
                    acc_ref(acc, i, c, q) = dz;
                }
#pragma unroll
                if (TXN == 16) {                             // two row groups share a warp
#pragma unroll
                    for (int h = 0; h < heads; ++h) sw[h] += __shfl_xor_sync(0xffffffffu, sw[h], 16);
                    sb += __shfl_xor_sync(0xffffffffu, sb, 16);
                }
                if ((tid & 31) < TXN) {
#pragma unroll
                    for (int h = 0; h < heads; ++h) scratch[(warp * 4 + h) * HID + j] = sw[h];
                    scratch[(warp * 4 + 3) * HID + j] = sb;
                }
#pragma unroll
                for (int i4 = 0; i4 < RT / 4; ++i4) {
                    float4 o;
                    o.x = acc_ref(acc, i4 * 4 + 0, c, q); o.y = acc_ref(acc, i4 * 4 + 1, c, q);
                    o.z = acc_ref(acc, i4 * 4 + 2, c, q); o.w = acc_ref(acc, i4 * 4 + 3, c, q);
                    *reinterpret_cast<float4*>(&sm.hT[j * H1_LD + ty * RT + i4 * 4]) = o;
                }
            }
        // dz2 to HBM in column blocks [4][mp][64]: the A operand of the dW2 kernel, one contiguous 4 KB tile per 16 rows
#pragma unroll
        for (int i = 0; i < RT; ++i)
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const float2 lo = acc[i][c * 2], hi = acc[i][c * 2 + 1];
                const int j0 = c * CSTR + tx * 4;
                *reinterpret_cast<float4*>(dz2b + ((int64_t)(j0 >> 6) * mp + row0 + ty * RT + i) * 64 + (j0 & 63)) = make_float4(lo.x, lo.y, hi.x, hi.y);
            }
    }
    __syncthreads();
    {
        const float* scratch = &sm.wt[0][0];
        float* dst = part_head + (int64_t)blockIdx.x * 4 * HID;
        for (int e = tid; e < 4 * HID; e += THREADS) {
            const int r = e / HID;
            if (r < heads || r == 3) {
                float t = scratch[e];
#pragma unroll
                for (int w = 1; w < NWARPS; ++w) t += scratch[w * 4 * HID + e];
                dst[e] = t;
            }
        }
    }
    __syncthreads();      // scratch consumed, dz2^T complete

    // ---------------- backward through layer 2: dh1 = dz2 W2, fc2.weight streamed in its torch layout ([j][k] is k-major)
    if (tid == 0) {
#pragma unroll
        for (int st = 0; st < NSTAGE; ++st) {
            mbar_expect_tx(&sm.full[st], KT * HID * 4);
            bulk_g2s(&sm.wt[st][0], w2 + st * KT * HID, KT * HID * 4, &sm.full[st]);
        }
    }
    acc_zero(acc);
#pragma unroll 1
    for (int t = 0; t < NT; ++t) {
        const int st = t & 1;
        mbar_wait(&sm.full[st], (t >> 1) & 1);               // NT/NSTAGE is even: the parity sequence restarts at 0
        tile_fma<KT>(acc, sm.hT + t * KT * H1_LD, H1_LD, &sm.wt[st][0], ty, tx);
        __syncthreads();
        if (tid == 0 && t + NSTAGE < NT) {
            mbar_expect_tx(&sm.full[st], KT * HID * 4);
            bulk_g2s(&sm.wt[st][0], w2 + (t + NSTAGE) * KT * HID, KT * HID * 4, &sm.full[st]);
        }
    }
    // dz1 = dh1 act'(h1) -> HBM row-major
#pragma unroll
    for (int i = 0; i < RT; ++i)
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const int64_t o = (row0 + ty * RT + i) * HID + c * CSTR + tx * 4;
            const float4 hv = *reinterpret_cast<const float4*>(h1g + o);
            const float2 lo = acc[i][c * 2], hi = acc[i][c * 2 + 1];
            *reinterpret_cast<float4*>(dz1g + o) = make_float4(lo.x * act_grad(hv.x, use_tanh), lo.y * act_grad(hv.y, use_tanh),
                                                              hi.x * act_grad(hv.z, use_tanh), hi.y * act_grad(hv.w, use_tanh));
        }
}
static_assert((HID / KT / NSTAGE) % 2 == 0, "mbarrier parity bookkeeping of the second streaming loop");

// ---------------------------------------------------------------------------------------------- dW2 = dz2^T h1
struct __align__(128) WgSmem {
    float a[WG_STAGES][KT * 64];     // dz2 tile  [16 rows][64 columns of one block]
    float b[WG_STAGES][KT * HID];    // h1 tile   [16 rows][256]
    uint64_t full[WG_STAGES];
};

__global__ void __launch_bounds__(THREADS, 2)
ppo_wgrad2_kernel(const float* __restrict__ dz2b, const float* __restrict__ h1g, int64_t mp, int slabs,
                  float* __restrict__ part_w2) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    WgSmem& sm = *reinterpret_cast<WgSmem*>(smem_raw);
    const int tid = threadIdx.x, tx = tid % TXN, ty = tid / TXN;
    const int jb = blockIdx.x, slab = blockIdx.y;
    const int64_t ktiles = mp / KT;
    const int64_t t0 = ktiles * slab / slabs, t1 = ktiles * (slab + 1) / slabs;
    const int nt = (int)(t1 - t0);
    const float* asrc = dz2b + ((int64_t)jb * mp + t0 * KT) * 64;
    const float* bsrc = h1g + t0 * KT * HID;
    if (tid == 0) {
#pragma unroll
        for (int st = 0; st < WG_STAGES; ++st) mbar_init(&sm.full[st], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        for (int st = 0; st < WG_STAGES && st < nt; ++st) {
            mbar_expect_tx(&sm.full[st], KT * 64 * 4 + KT * HID * 4);
            bulk_g2s(&sm.a[st][0], asrc + (int64_t)st * KT * 64, KT * 64 * 4, &sm.full[st]);
            bulk_g2s(&sm.b[st][0], bsrc + (int64_t)st * KT * HID, KT * HID * 4, &sm.full[st]);
        }
    }
    float2 acc[RT][NP];
    acc_zero(acc);
#pragma unroll 1
    for (int t = 0; t < nt; ++t) {
        const int st = t % WG_STAGES;
        mbar_wait(&sm.full[st], (t / WG_STAGES) & 1);
        tile_fma<KT>(acc, &sm.a[st][0], 64, &sm.b[st][0], ty, tx);
        __syncthreads();
        if (tid == 0 && t + WG_STAGES < nt) {
            mbar_expect_tx(&sm.full[st], KT * 64 * 4 + KT * HID * 4);
            bulk_g2s(&sm.a[st][0], asrc + (int64_t)(t + WG_STAGES) * KT * 64, KT * 64 * 4, &sm.full[st]);
            bulk_g2s(&sm.b[st][0], bsrc + (int64_t)(t + WG_STAGES) * KT * HID, KT * HID * 4, &sm.full[st]);
        }
    }
    float* dst = part_w2 + (int64_t)slab * HID * HID;        // [j][k] = fc2.weight layout
#pragma unroll
    for (int i = 0; i < RT; ++i)
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const float2 lo = acc[i][c * 2], hi = acc[i][c * 2 + 1];
            *reinterpret_cast<float4*>(dst + (int64_t)(jb * 64 + ty * RT + i) * HID + c * CSTR + tx * 4) = make_float4(lo.x, lo.y, hi.x, hi.y);
        }
}

// ---------------------------------------------------------------------------------------------- dW1 = dz1^T x, db1
// A streaming pass: 16-row tiles of dz1 (16 KB, contiguous) and of the gathered observations (2 KB) arrive through a
// 3-stage TMA pipeline; thread j owns row j of fc1.weight's gradient.
constexpr int W1_STAGES = 3;
struct __align__(128) W1Smem {
    float z[W1_STAGES][KT * HID];
    float x[W1_STAGES][KT * XS_LD];
    uint64_t full[W1_STAGES];
};

__global__ void __launch_bounds__(HID, 4)
ppo_wgrad1_kernel(const float* __restrict__ dz1g, const float* __restrict__ xs, int64_t mp, int slabs,
                  float* __restrict__ part_w1, float* __restrict__ part_b1) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    W1Smem& sm = *reinterpret_cast<W1Smem*>(smem_raw);
    const int j = threadIdx.x, slab = blockIdx.x;
    const int64_t ktiles = mp / KT;
    const int64_t t0 = ktiles * slab / slabs, t1 = ktiles * (slab + 1) / slabs;
    const int nt = (int)(t1 - t0);
    const float* zsrc = dz1g + t0 * KT * HID;
    const float* xsrc = xs + t0 * KT * XS_LD;
    if (j == 0) {
#pragma unroll
        for (int st = 0; st < W1_STAGES; ++st) mbar_init(&sm.full[st], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (j == 0) {
        for (int st = 0; st < W1_STAGES && st < nt; ++st) {
            mbar_expect_tx(&sm.full[st], KT * HID * 4 + KT * XS_LD * 4);
            bulk_g2s(&sm.z[st][0], zsrc + (int64_t)st * KT * HID, KT * HID * 4, &sm.full[st]);
            bulk_g2s(&sm.x[st][0], xsrc + (int64_t)st * KT * XS_LD, KT * XS_LD * 4, &sm.full[st]);
        }
    }
    float acc[IN], sb = 0.0f;
#pragma unroll
    for (int d = 0; d < IN; ++d) acc[d] = 0.0f;
#pragma unroll 1
    for (int t = 0; t < nt; ++t) {
        const int st = t % W1_STAGES;
        mbar_wait(&sm.full[st], (t / W1_STAGES) & 1);
#pragma unroll 4
        for (int r = 0; r < KT; ++r) {
            const float z = sm.z[st][r * HID + j];
            const float4* xr = reinterpret_cast<const float4*>(&sm.x[st][r * XS_LD]);
            float x[20];
#pragma unroll
            for (int v = 0; v < 5; ++v) { const float4 q = xr[v]; x[v * 4] = q.x; x[v * 4 + 1] = q.y; x[v * 4 + 2] = q.z; x[v * 4 + 3] = q.w; }
            sb += z;
#pragma unroll
            for (int d = 0; d < IN; ++d) acc[d] = fmaf(z, x[d], acc[d]);
        }
        __syncthreads();
        if (j == 0 && t + W1_STAGES < nt) {
            mbar_expect_tx(&sm.full[st], KT * HID * 4 + KT * XS_LD * 4);
            bulk_g2s(&sm.z[st][0], zsrc + (int64_t)(t + W1_STAGES) * KT * HID, KT * HID * 4, &sm.full[st]);
            bulk_g2s(&sm.x[st][0], xsrc + (int64_t)(t + W1_STAGES) * KT * XS_LD, KT * XS_LD * 4, &sm.full[st]);
        }
    }
    float* dst = part_w1 + (int64_t)slab * HID * IN + j * IN;       // fc1.weight layout [j][18]
#pragma unroll
    for (int d = 0; d < IN; ++d) dst[d] = acc[d];
    part_b1[(int64_t)slab * HID + j] = sb;
}

// ---------------------------------------------------------------------------------------------- partial sums -> flat gradient
// block = 32 consecutive elements x 32 groups of partials; fixed summation order (deterministic gradients)
struct SumGroup { const float* src; int64_t stride; int parts, elems, dst_off, block0; };
struct SumPlan { SumGroup g[6]; int groups; };

__global__ void __launch_bounds__(1024)
colsum_kernel(const SumPlan plan, float* __restrict__ grads) {
    __shared__ float red[32][33];
    int gi = 0;
#pragma unroll
    for (int k = 1; k < 6; ++k) if (k < plan.groups && (int)blockIdx.x >= plan.g[k].block0) gi = k;
    const SumGroup g = plan.g[gi];
    const int lane = threadIdx.x & 31, ps = threadIdx.x >> 5;
    const int e = ((int)blockIdx.x - g.block0) * 32 + lane;
    float sum = 0.0f;
    if (e < g.elems) {
        const float* src = g.src + e;
#pragma unroll 8
        for (int p = ps; p < g.parts; p += 32) sum += src[(int64_t)p * g.stride];
    }
    red[ps][lane] = sum;
    __syncthreads();
    if (ps == 0 && e < g.elems) {
        float t = 0.0f;
#pragma unroll
        for (int k = 0; k < 32; ++k) t += red[k][lane];
        grads[g.dst_off + e] = t;
    }
}

// ---------------------------------------------------------------------------------------------- clip + Adam + repack
constexpr int ADAM_CTAS = 8, ADAM_THREADS = 1024, ADAM_PER = 9;
static_assert(ADAM_CTAS * ADAM_THREADS * ADAM_PER >= SAT_PPO_PARAM_FLOATS(3), "one pass must cover every parameter");

__device__ __forceinline__ int packed_index(int i, int heads) {
    if (i < SAT_PPO_OFF_B1) { const int j = i / IN, k = i - j * IN; return OFF_W1T + k * HID + j; }
    if (i < SAT_PPO_OFF_W2) return OFF_B1 + (i - SAT_PPO_OFF_B1);
    if (i < SAT_PPO_OFF_B2) { const int r = i - SAT_PPO_OFF_W2; const int j = r / HID, k = r - j * HID; return OFF_W2T + k * HID + j; }
    if (i < SAT_PPO_OFF_W3) return OFF_B2 + (i - SAT_PPO_OFF_B2);
    const int b3 = off_b3(heads);
    if (i < b3) return OFF_W3 + (i - SAT_PPO_OFF_W3);
    if (i < b3 + heads) return OFF_B3 + (i - b3);
    return OFF_LS + (i - b3 - heads);
}

// STATS: before the update, thread 0 adds the minibatch's global means (loss slot grads[total] and, for the actor, the
// diagnostics tail grads[total + 2 ..]; summed over the peers in rank order on the peer path, times grad_scale), the pre-clip
// gradient norm, the clip coefficient and a count of 1 to record[SAT_PPO_STATS_DOUBLES] (fp64)
template <bool STATS>
__global__ void __cluster_dims__(ADAM_CTAS, 1, 1) __launch_bounds__(ADAM_THREADS)
ppo_adam_kernel(float* __restrict__ params, float* __restrict__ packed, const float* __restrict__ grads,
                float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq, int heads, const float* __restrict__ lr_ptr,
                float beta1, float beta2, float eps, float max_norm, float grad_scale, int64_t* __restrict__ step_ptr,
                const float* const* __restrict__ peers, int world, int64_t peer_off, double* __restrict__ record) {
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ float warp_sums[32];
    __shared__ float cta_sum;
    const int total = param_floats(heads);
    const int gtid = blockIdx.x * ADAM_THREADS + threadIdx.x;
    float g[ADAM_PER], ss = 0.0f;
#pragma unroll
    for (int k = 0; k < ADAM_PER; ++k) {
        const int i = gtid + k * ADAM_CTAS * ADAM_THREADS;
        float gi = 0.0f;
        if (i < total) {
            if (peers) {
                // gradient all-reduce fused into the optimiser step: every rank reads all ranks' flat gradients from
                // NVLink peer memory (symmetric allocation) and adds them in rank order, so the replicas stay bit-identical
                for (int r = 0; r < world; ++r) gi += __ldcg(peers[r] + peer_off + i);
            } else {
                gi = grads[i];
            }
        }
        g[k] = gi * grad_scale;
        ss = fmaf(g[k], g[k], ss);
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = warp_sums[threadIdx.x];
#pragma unroll
        for (int off = 16; off; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (threadIdx.x == 0) cta_sum = t;
    }
    cluster.sync();
    float sumsq = 0.0f;
#pragma unroll
    for (int r = 0; r < ADAM_CTAS; ++r) sumsq += *cluster.map_shared_rank(&cta_sum, r);     // same order in every CTA
    const int64_t step = *step_ptr + 1;
    cluster.sync();                                           // nobody leaves (or bumps the step) while peers still read
    float coef = 1.0f;
    if (max_norm > 0.0f) coef = fminf(max_norm / (sqrtf(sumsq) + 1e-6f), 1.0f);               // clip_grad_norm_ (:229, :238)
    if constexpr (STATS) {
        if (gtid == 0) {
            auto slot = [&](int k) {
                float v = 0.0f;
                if (peers) { for (int r = 0; r < world; ++r) v += __ldcg(peers[r] + peer_off + total + k); }
                else v = grads[total + k];
                return (double)(v * grad_scale);
            };
            record[SAT_PPO_STAT_LOSS] += slot(0);
            if (heads == 3) {
                record[SAT_PPO_STAT_SURROGATE] += slot(2);
                record[SAT_PPO_STAT_ENTROPY] += slot(3);
                record[SAT_PPO_STAT_APPROX_KL] += slot(4);
                record[SAT_PPO_STAT_CLIP_FRAC] += slot(5);
            }
            record[SAT_PPO_STAT_GRAD_NORM] += (double)sqrtf(sumsq);
            record[SAT_PPO_STAT_CLIP_COEF] += (double)coef;
            record[SAT_PPO_STAT_COUNT] += 1.0;
        }
    }
    const float lr = *lr_ptr;
    const float bc1 = 1.0f - powf(beta1, (float)step), bc2 = 1.0f - powf(beta2, (float)step);
    const float step_size = lr / bc1, bc2_sqrt = sqrtf(bc2);
#pragma unroll
    for (int k = 0; k < ADAM_PER; ++k) {
        const int i = gtid + k * ADAM_CTAS * ADAM_THREADS;
        if (i < total) {
            const float gr = g[k] * coef;
            float m = exp_avg[i], v = exp_avg_sq[i];
            m = m + (gr - m) * (1.0f - beta1);                                                // exp_avg.lerp_(grad, 1 - beta1)
            v = v * beta2 + (1.0f - beta2) * gr * gr;
            const float denom = sqrtf(v) / bc2_sqrt + eps;
            const float p = params[i] - step_size * (m / denom);
            exp_avg[i] = m; exp_avg_sq[i] = v; params[i] = p;
            packed[packed_index(i, heads)] = p;
        }
    }
    if (gtid == 0) *step_ptr = step;
}

__global__ void ppo_pack_kernel(const float* __restrict__ params, float* __restrict__ packed, int heads) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < param_floats(heads)) packed[packed_index(i, heads)] = params[i];
}
__global__ void ppo_pack_zero_kernel(float* __restrict__ packed) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= OFF_W3 && i < PACKED_FLOATS) packed[i] = 0.0f;
}

inline int launch_status() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? SAT_OK : (int)e;
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return e == cudaSuccess ? SAT_OK : (int)e;
}

int check_net(const SatPpoNet* net) {
    if (!net || !net->params || !net->packed || !net->grads || !net->exp_avg || !net->exp_avg_sq || !net->workspace) return SAT_ERR_NULL;
    if (net->heads != 1 && net->heads != 3) return SAT_ERR_SIZE;
    if (((uintptr_t)net->params | (uintptr_t)net->packed | (uintptr_t)net->workspace | (uintptr_t)net->grads) & 15) return SAT_ERR_SIZE;
    return SAT_OK;
}

// everything after the forward/backward kernel: weight-gradient kernels and the partial sums
int finish_grads(const SatPpoNet* net, const Workspace& w, cudaStream_t stream, int64_t head_tiles, bool tc) {
    const int heads = net->heads;
    const int64_t ktiles = w.mp / KT;
    const int slabs1 = (int)(w.mp / 16 < W1_SLABS ? w.mp / 16 : W1_SLABS);
    int rc;
    int slabs2 = (int)(ktiles < W2_SLABS ? ktiles : W2_SLABS);
    if (tc) {
        const int64_t chunks = w.mp / 32;
        slabs2 = (int)(chunks < W2_SLABS ? chunks : W2_SLABS);
        rc = ppo_wgrad2_tc_launch(w.dz2b, w.h1, w.mp, slabs2, w.part_w2, stream);
        if (rc) return rc;
    } else {
        rc = set_smem(ppo_wgrad2_kernel, sizeof(WgSmem));
        if (rc) return rc;
        ppo_wgrad2_kernel<<<dim3(4, slabs2), THREADS, sizeof(WgSmem), stream>>>(w.dz2b, w.h1, w.mp, slabs2, w.part_w2);
    }
    rc = set_smem(ppo_wgrad1_kernel, sizeof(W1Smem));
    if (rc) return rc;
    ppo_wgrad1_kernel<<<slabs1, HID, sizeof(W1Smem), stream>>>(w.dz1, w.xs, w.mp, slabs1, w.part_w1, w.part_b1);
    SumPlan plan;
    int nb = 0, gi = 0;
    auto add = [&](const float* src, int64_t stride, int parts, int elems, int dst_off) {
        plan.g[gi] = SumGroup{src, stride, parts, elems, dst_off, nb};
        nb += (elems + 31) / 32; ++gi;
    };
    add(w.part_w2, (int64_t)HID * HID, slabs2, HID * HID, SAT_PPO_OFF_W2);
    add(w.part_w1, (int64_t)HID * IN, slabs1, HID * IN, SAT_PPO_OFF_W1);
    add(w.part_b1, HID, slabs1, HID, SAT_PPO_OFF_B1);
    add(w.part_head, 4 * HID, (int)head_tiles, heads * HID, SAT_PPO_OFF_W3);
    add(w.part_head + 3 * HID, 4 * HID, (int)head_tiles, HID, SAT_PPO_OFF_B2);
    add(w.part_scal, 8, (int)head_tiles, heads == 3 ? 7 : 2, off_b3(heads));        // db3, dlog_std, loss (one past the parameters)
    plan.groups = gi;
    colsum_kernel<<<nb, 1024, 0, stream>>>(plan, net->grads);
    return launch_status();
}

// forward / backward kernel: tensor cores (ppo_fb_tc.cu, default) or fp32 FFMA2 (ppo_fb_kernel); SAT_PPO_TC=0 or
// sat_ppo_use_tensor_cores(0) selects the latter
int g_ppo_tc = -1;
inline bool ppo_tc_enabled() {
    if (g_ppo_tc < 0) { const char* e = std::getenv("SAT_PPO_TC"); g_ppo_tc = (e && e[0] == '0') ? 0 : 1; }
    return g_ppo_tc != 0;
}

// the per-tile diagnostics -> grads[n + 2 .. n + 6), the tail the gradient exchange carries with the gradient
int sum_stats(const SatPpoNet* net, const Workspace& w, cudaStream_t stream, int64_t head_tiles) {
    SumPlan plan;
    plan.g[0] = SumGroup{w.part_stat, 8, (int)head_tiles, 4, param_floats(net->heads) + 2, 0};
    plan.groups = 1;
    colsum_kernel<<<1, 1024, 0, stream>>>(plan, net->grads);
    return launch_status();
}

template <bool STATS>
int actor_grad(const SatPpoNet* net, const float* s, const float* a, const float* old_logp, const float* adv,
               const int64_t* index, int64_t mb, float epsilon, float entropy_coef, cudaStream_t stream) {
    int rc = check_net(net);
    if (rc) return rc;
    if (!s || !a || !old_logp || !adv) return SAT_ERR_NULL;
    if (net->heads != 3 || mb <= 0) return SAT_ERR_SIZE;
    rc = set_smem(ppo_fb_kernel<false, STATS>, STATS ? sizeof(FbSmemStats) : sizeof(FbSmem));
    if (rc) return rc;
    const Workspace w = ws_carve(net->workspace, mb);
    float* part_stat = STATS ? w.part_stat : nullptr;
    if (ppo_tc_enabled()) {
        rc = ppo_fb_tc_launch(false, net->use_tanh != 0, net->packed, w.tc_image, net->max_action, s, a, old_logp, adv, nullptr, index, mb,
                              1.0f / (float)mb, epsilon, entropy_coef, w.h1, w.dz2b, w.dz1, w.xs, w.part_head, w.part_scal, w.mp,
                              part_stat, stream);
        if (rc) return rc;
        rc = finish_grads(net, w, stream, w.mp / MP_ALIGN, true);
        if (rc || !STATS) return rc;
        return sum_stats(net, w, stream, w.mp / MP_ALIGN);
    }
    ppo_fb_kernel<false, STATS><<<(unsigned)w.tiles, THREADS, STATS ? sizeof(FbSmemStats) : sizeof(FbSmem), stream>>>(
        net->packed, net->params + SAT_PPO_OFF_W2, net->use_tanh, net->max_action, s, a, old_logp, adv, nullptr, index, mb,
        1.0f / (float)mb, epsilon, entropy_coef, w.h1, w.dz2b, w.dz1, w.xs, w.part_head, w.part_scal, w.mp, part_stat);
    rc = launch_status();
    if (rc) return rc;
    rc = finish_grads(net, w, stream, w.tiles, false);
    if (rc || !STATS) return rc;
    return sum_stats(net, w, stream, w.tiles);
}

template <bool STATS>
int adam(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm, float grad_scale,
         int64_t* step, bool peer_path, const float* const* peer_grads, int world, int64_t offset_floats, double* record,
         cudaStream_t stream) {
    int rc = check_net(net);
    if (rc) return rc;
    if (!lr || !step || (peer_path && !peer_grads) || (STATS && !record)) return SAT_ERR_NULL;
    if (peer_path && (world < 1 || world > 64 || offset_floats < 0)) return SAT_ERR_SIZE;
    ppo_adam_kernel<STATS><<<ADAM_CTAS, ADAM_THREADS, 0, stream>>>(net->params, net->packed, net->grads, net->exp_avg,
                                                                  net->exp_avg_sq, net->heads, lr, beta1, beta2, eps,
                                                                  max_grad_norm, grad_scale, step, peer_grads, world,
                                                                  offset_floats, record);
    return launch_status();
}

}  // namespace

extern "C" {

int sat_ppo_use_tensor_cores(int enable) {
    const int prev = ppo_tc_enabled() ? 1 : 0;
    if (enable >= 0) g_ppo_tc = enable ? 1 : 0;
    return prev;
}

int64_t sat_ppo_workspace_floats(int64_t mb) { return mb > 0 ? ws_floats(mb) : 0; }

int sat_ppo_pack(const SatPpoNet* net, void* stream) {
    int rc = check_net(net);
    if (rc) return rc;
    ppo_pack_zero_kernel<<<(PACKED_FLOATS + 255) / 256, 256, 0, (cudaStream_t)stream>>>(net->packed);
    ppo_pack_kernel<<<(param_floats(net->heads) + 255) / 256, 256, 0, (cudaStream_t)stream>>>(net->params, net->packed, net->heads);
    return launch_status();
}

int sat_ppo_actor_grad(const SatPpoNet* net, const float* s, const float* a, const float* old_logp, const float* adv,
                       const int64_t* index, int64_t mb, float epsilon, float entropy_coef, void* stream) {
    return actor_grad<false>(net, s, a, old_logp, adv, index, mb, epsilon, entropy_coef, (cudaStream_t)stream);
}

int sat_ppo_actor_grad_stats(const SatPpoNet* net, const float* s, const float* a, const float* old_logp, const float* adv,
                             const int64_t* index, int64_t mb, float epsilon, float entropy_coef, void* stream) {
    return actor_grad<true>(net, s, a, old_logp, adv, index, mb, epsilon, entropy_coef, (cudaStream_t)stream);
}

int sat_ppo_critic_grad(const SatPpoNet* net, const float* s, const float* v_target, const int64_t* index, int64_t mb,
                        void* stream) {
    int rc = check_net(net);
    if (rc) return rc;
    if (!s || !v_target) return SAT_ERR_NULL;
    if (net->heads != 1 || mb <= 0) return SAT_ERR_SIZE;
    rc = set_smem(ppo_fb_kernel<true, false>, sizeof(FbSmem));
    if (rc) return rc;
    const Workspace w = ws_carve(net->workspace, mb);
    if (ppo_tc_enabled()) {
        rc = ppo_fb_tc_launch(true, net->use_tanh != 0, net->packed, w.tc_image, 0.0f, s, nullptr, nullptr, nullptr, v_target, index, mb,
                              1.0f / (float)mb, 0.0f, 0.0f, w.h1, w.dz2b, w.dz1, w.xs, w.part_head, w.part_scal, w.mp,
                              nullptr, (cudaStream_t)stream);
        if (rc) return rc;
        return finish_grads(net, w, (cudaStream_t)stream, w.mp / MP_ALIGN, true);
    }
    ppo_fb_kernel<true, false><<<(unsigned)w.tiles, THREADS, sizeof(FbSmem), (cudaStream_t)stream>>>(
        net->packed, net->params + SAT_PPO_OFF_W2, net->use_tanh, 0.0f, s, nullptr, nullptr, nullptr, v_target, index, mb,
        1.0f / (float)mb, 0.0f, 0.0f, w.h1, w.dz2b, w.dz1, w.xs, w.part_head, w.part_scal, w.mp, nullptr);
    rc = launch_status();
    if (rc) return rc;
    return finish_grads(net, w, (cudaStream_t)stream, w.tiles, false);
}

int sat_ppo_adam(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm,
                 float grad_scale, int64_t* step, void* stream) {
    return adam<false>(net, lr, beta1, beta2, eps, max_grad_norm, grad_scale, step, false, nullptr, 1, 0, nullptr, (cudaStream_t)stream);
}

int sat_ppo_adam_stats(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm,
                       float grad_scale, int64_t* step, double* record, void* stream) {
    return adam<true>(net, lr, beta1, beta2, eps, max_grad_norm, grad_scale, step, false, nullptr, 1, 0, record, (cudaStream_t)stream);
}

int sat_ppo_adam_peers(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm,
                       float grad_scale, int64_t* step, const float* const* peer_grads, int world, int64_t offset_floats,
                       void* stream) {
    return adam<false>(net, lr, beta1, beta2, eps, max_grad_norm, grad_scale, step, true, peer_grads, world, offset_floats, nullptr,
                       (cudaStream_t)stream);
}

int sat_ppo_adam_peers_stats(const SatPpoNet* net, const float* lr, float beta1, float beta2, float eps, float max_grad_norm,
                             float grad_scale, int64_t* step, const float* const* peer_grads, int world, int64_t offset_floats,
                             double* record, void* stream) {
    return adam<true>(net, lr, beta1, beta2, eps, max_grad_norm, grad_scale, step, true, peer_grads, world, offset_floats, record,
                      (cudaStream_t)stream);
}

}  // extern "C"
