// ppo_fb_tc.cu -- the forward / backward kernel of the fused PPO minibatch step on the tensor cores (sm_100a).
//
// Reference behaviour replaced: the same as ppo_fb_kernel in ppo_update.cu (the body of the K-epoch loop of
// PPO_continuous.update, ppo_continuous.py:216-239: actor / critic forward, clipped-surrogate + entropy / MSE loss, backward
// down to dz1), which the reference evaluates in fp32.
//
// The three 128 x 256 x {18, 256, 256} contractions per row tile (h1 = act(W1 x), h2 = act(W2 h1), dh1 = dz2 W2) run as exact
// bf16x3 splits on tcgen05.mma with the accumulators in TMEM - the scheme of actor_tc.cu (six bf16 word products per fp32
// product, the exact 16-bit A_h B_h products in their own accumulator), so the gradients keep fp32-level accuracy
// (tests/test_gpu_ppo_fused.py compares them with PyTorch autograd). Same outputs and layouts as ppo_fb_kernel, so the
// weight-gradient kernels, the partial sums and the Adam kernel of ppo_update.cu are unchanged:
//   h1 [mp][256], dz2 in column blocks [4][mp][64], dz1 [mp][256], xs [mp][32] (gathered observations), per-tile partial sums
//   part_head [tile][4][256] (dW3 rows, db2) and part_scal [tile][8] (db3, dlog_std, loss); a tile is 128 rows here.
//
// Persistent kernel, one CTA per SM, 576 threads: 16 row warps (thread = row r = tid & 127, quarter p = tid >> 7), one MMA-issue
// lane, one weight-stream lane. Per tile the A ring (4 stages, FIFO) carries 17 operand chunks - the gathered observations, the
// eight chunks of h1, the eight chunks of dz2 - and the B ring (4 stages) the 34 matching weight sub-chunks of the image
// (W1, W2 for the forward, W2 transposed for the backward). The K order of the backward product is permuted (chunk kc holds
// columns 64 p + 8 kc + j of dz2) so that every row thread writes one 16-byte piece of every chunk, exactly like the forward.
// TMEM: [0, 256) A_h B_h, [256, 512) the small products; the three products of a tile reuse the same columns one after the other.
#include <cstdint>
#include <cuda_runtime.h>
#include "tc_mlp.cuh"
#include "ppo_fb_tc.cuh"

namespace {
using namespace mlp;
using namespace tcm;

constexpr int FB_CHUNKS = 1 + 2 * NCH;           // A chunks per tile: x, h1 x 8, dz2 x 8
constexpr int FB_SUBS = FB_CHUNKS * NSUB;        // weight sub-chunks per tile: 34
static_assert(FB_SUBS * B_STAGE == SAT_PPO_TC_IMAGE_BYTES, "header constant out of sync");
constexpr int XS_LD = 32;
constexpr int FNSA = 3, FNSB = 3;                // ring depths (the tensor core is not this kernel's limit; the shared memory goes to the staging below)
constexpr int ST_LD = 20;                        // staging row: 16 floats + 4 of padding (conflict-free 16-byte accesses)
constexpr int ST_WARP = 32 * ST_LD;              // floats per row warp
constexpr int OFF_A = 0;
constexpr int OFF_B = OFF_A + FNSA * A_STAGE;
constexpr int OFF_STG = OFF_B + FNSB * B_STAGE;  // per-warp transposition staging for the row-major HBM stores / loads
constexpr int OFF_RED = OFF_STG + 16 * ST_WARP * 4;   // head partial sums [NPART][TM] float4
constexpr int OFF_DZ3 = OFF_RED + NPART * TM * 16;   // per-row head gradients [TM] float4
constexpr int OFF_COL = OFF_DZ3 + TM * 16;       // column partial sums [16 warps][4][64]
constexpr int OFF_SCAL = OFF_COL + 16 * 4 * 64 * 4;  // per-warp scalar partial sums [4][8]
constexpr int SM_W3T = OFF_SCAL + 4 * 8 * 4;     // float4 [HID]: (W3[0][c], W3[1][c], W3[2][c], b2[c] (x 2 log2 e for tanh))
constexpr int OFF_B1P = SM_W3T + HID * 16;       // b1 in layer-1 accumulator column order (x 2 log2 e for tanh)
constexpr int OFF_BAR = OFF_B1P + HID * 4;
constexpr int OFF_TMEM = OFF_BAR + 24 * 8;
constexpr int FB_SMEM = OFF_TMEM + 16 + 1024;
constexpr int OFF_STAT = OFF_TMEM + 16;          // stats instantiation only: per-warp partial sums of the diagnostics [4][4]
constexpr int FB_SMEM_STATS = FB_SMEM + 4 * 4 * 4;
static_assert(FB_SMEM_STATS <= 227 * 1024, "shared memory budget");

// image: chunk 0 = W1 (as in actor_tc.cu), chunks 1..8 = W2 forward (n = output unit j, k = input unit), chunks 9..16 = W2
// backward (n = input unit i, k = output unit j in the permuted order: position kk = 8 p + jj of chunk kc is j = 64 p + 8 kc + jj)
__global__ void ppo_fb_tc_pack_kernel(const float* __restrict__ packed, unsigned char* __restrict__ image) {
    asm volatile("griddepcontrol.launch_dependents;");                  // see actor_tc_pack_kernel
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= FB_CHUNKS * 4 * HID) return;
    const int n = idx % HID, c16 = (idx / HID) & 3, chunk = idx / (4 * HID);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int kk = c16 * 8 + j;
        if (chunk == 0) v[j] = (kk < IN) ? packed[OFF_W1T + kk * HID + l1_unit(n)] : 0.0f;
        else if (chunk <= NCH) v[j] = packed[OFF_W2T + ((chunk - 1) * KC + kk) * HID + n];
        else v[j] = packed[OFF_W2T + n * HID + 64 * c16 + 8 * (chunk - 1 - NCH) + j];      // fc2.weight[j][i], i = n
    }
    uint4 H, M, L;
    split8(v, H, M, L);
    unsigned char* base = image + (size_t)(chunk * NSUB + (c16 >> 1)) * B_STAGE + sw32((uint32_t)n, (uint32_t)(c16 & 1));
    *reinterpret_cast<uint4*>(base) = H;
    *reinterpret_cast<uint4*>(base + B_WORD) = M;
    *reinterpret_cast<uint4*>(base + 2 * B_WORD) = L;
}

// transposing warp reduction: every lane holds 16 values; afterwards lane l holds, in v[0], the sum over the 32 lanes of value
// l >> 1 (both lanes of a pair hold the same sum). 16 shuffles.
__device__ __forceinline__ void warp_transpose_sum16(float (&v)[16], int lane) {
#pragma unroll
    for (int off = 16, n = 16; off >= 2; off >>= 1, n >>= 1) {
        const bool up = lane & off;
#pragma unroll
        for (int i = 0; i < n / 2; ++i) {
            const float send = up ? v[i] : v[i + n / 2];
            const float keep = up ? v[i + n / 2] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}

#ifdef SAT_TC_TRACE
__device__ unsigned long long g_fb_trace[256];
__device__ __forceinline__ void fb_trace(int slot) {
    if (blockIdx.x == 0 && threadIdx.x == 0 && slot < 256) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); g_fb_trace[slot] = t; }
}
#define FB_TRACE(slot) fb_trace(slot)
#else
#define FB_TRACE(slot)
#endif

// A row thread holds 64 values of ITS row; written straight to a row-major buffer, every store instruction of a warp would touch
// 32 rows x 16 bytes (half-used sectors in 32 different lines: 9 us per 128 x 256 tile, measured). These helpers pass 16 values
// per row at a time through a per-warp staging tile so that each instruction moves whole 32 / 64-byte row segments.
// v[b * 16 + q * 4 + e] goes to gwarp[row * row_stride + seg_off(b, q) + e]: seg(b, q) = float offset of 16-byte piece q of batch b.
template <class SegOff>
__device__ __forceinline__ void store_rows_batch(int b, float* __restrict__ gwarp, int64_t row_stride, const float (&v)[64], float* st, int lane, SegOff seg) {
#pragma unroll
    for (int q = 0; q < 4; ++q)
        *reinterpret_cast<float4*>(st + lane * ST_LD + q * 4) = make_float4(v[b * 16 + q * 4], v[b * 16 + q * 4 + 1], v[b * 16 + q * 4 + 2], v[b * 16 + q * 4 + 3]);
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int idx = i * 32 + lane, rr = idx >> 2, pc = idx & 3;
        *reinterpret_cast<float4*>(gwarp + rr * row_stride + seg(b, pc)) = *reinterpret_cast<const float4*>(st + rr * ST_LD + pc * 4);
    }
    __syncwarp();
}
template <class SegOff>
__device__ __forceinline__ void store_rows(float* __restrict__ gwarp, int64_t row_stride, const float (&v)[64], float* st, int lane, SegOff seg) {
#pragma unroll
    for (int b = 0; b < 4; ++b) store_rows_batch(b, gwarp, row_stride, v, st, lane, seg);
}
// v[b * 16 + q * 4 + e] *= act'(g[row][seg(b, q) + e]) with the same access pattern (g = h1)
template <bool TANH, class SegOff>
__device__ __forceinline__ void scale_by_act_grad(const float* __restrict__ gwarp, int64_t row_stride, float (&v)[64], float* st, int lane, SegOff seg);

template <bool TANH>
__device__ __forceinline__ float act_grad_of(float h) { return TANH ? 1.0f - h * h : (h > 0.0f ? 1.0f : 0.0f); }

template <bool TANH, class SegOff>
__device__ __forceinline__ void scale_by_act_grad(const float* __restrict__ gwarp, int64_t row_stride, float (&v)[64], float* st, int lane, SegOff seg) {
#pragma unroll
    for (int b = 0; b < 4; ++b) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = i * 32 + lane, rr = idx >> 2, pc = idx & 3;
            *reinterpret_cast<float4*>(st + rr * ST_LD + pc * 4) = *reinterpret_cast<const float4*>(gwarp + rr * row_stride + seg(b, pc));
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 h = *reinterpret_cast<const float4*>(st + lane * ST_LD + q * 4);
            v[b * 16 + q * 4] *= act_grad_of<TANH>(h.x); v[b * 16 + q * 4 + 1] *= act_grad_of<TANH>(h.y);
            v[b * 16 + q * 4 + 2] *= act_grad_of<TANH>(h.z); v[b * 16 + q * 4 + 3] *= act_grad_of<TANH>(h.w);
        }
        __syncwarp();
    }
}

// STATS (actor only): the row threads also reduce the per-row diagnostics (surrogate, entropy, approximate KL, clipped), each
// scaled by inv_n like the loss, into part_stat [tile][8] (the first four entries)
template <bool CRITIC, bool TANH, bool STATS>
__global__ void __launch_bounds__(TC_THREADS, 1)
ppo_fb_tc_kernel(const float* __restrict__ packed, const unsigned char* __restrict__ image, float max_action,
                 const float* __restrict__ s, const float* __restrict__ a, const float* __restrict__ old_logp,
                 const float* __restrict__ adv, const float* __restrict__ v_target, const int64_t* __restrict__ index,
                 int64_t n, float inv_n, float epsilon, float entropy_coef,
                 float* __restrict__ h1g, float* __restrict__ dz2b, float* __restrict__ dz1g, float* __restrict__ xs,
                 float* __restrict__ part_head, float* __restrict__ part_scal, int64_t mp, float* __restrict__ part_stat) {
    static_assert(!(STATS && CRITIC), "the critic has no per-row diagnostics beyond its loss");
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* sm = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    float* stg = reinterpret_cast<float*>(sm + OFF_STG);
    float4* red = reinterpret_cast<float4*>(sm + OFF_RED);
    float4* dz3s = reinterpret_cast<float4*>(sm + OFF_DZ3);
    float* colp = reinterpret_cast<float*>(sm + OFF_COL);
    float* scal = reinterpret_cast<float*>(sm + OFF_SCAL);
    float4* w3t = reinterpret_cast<float4*>(sm + SM_W3T);
    float* b1p = reinterpret_cast<float*>(sm + OFF_B1P);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + OFF_BAR);
    uint64_t* b_full = bars;
    uint64_t* b_empty = bars + FNSB;
    uint64_t* a_full = bars + 2 * FNSB;
    uint64_t* a_empty = a_full + FNSA;
    uint64_t* l1_full = a_empty + FNSA;        // layer-1 accumulators complete
    uint64_t* l1_read = l1_full + 1;          // ... and read by every row
    uint64_t* l2_full = l1_full + 2;          // layer-2 accumulators complete
    uint64_t* l2_read = l1_full + 3;
    uint64_t* l3_full = l1_full + 4;          // dh1 accumulators complete
    uint64_t* acc_free = l1_full + 5;         // ... and read: the next tile's layer 1 may start
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + OFF_TMEM);
    const int tid = threadIdx.x, warp = tid >> 5;
    constexpr int heads = CRITIC ? 1 : 3;
    const int ntiles = (int)(mp / TM);
    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;     // >= 1: gridDim.x <= ntiles

    if (tid == 0) {
        for (int i = 0; i < FNSB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
        for (int i = 0; i < FNSA; ++i) { mbar_init(&a_full[i], TC_COMPUTE / 32); mbar_init(&a_empty[i], 1); }
        mbar_init(l1_full, 1); mbar_init(l1_read, TC_COMPUTE / 32);
        mbar_init(l2_full, 1); mbar_init(l2_read, TC_COMPUTE / 32);
        mbar_init(l3_full, 1); mbar_init(acc_free, TC_COMPUTE / 32);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == TC_COMPUTE / 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int c = tid; c < HID; c += TC_THREADS) {
        const float bs = TANH ? kTwoLog2e : 1.0f;
        b1p[c] = packed[OFF_B1 + l1_unit(c)] * bs;
        w3t[c] = make_float4(packed[OFF_W3 + c], heads > 1 ? packed[OFF_W3 + HID + c] : 0.0f, heads > 1 ? packed[OFF_W3 + 2 * HID + c] : 0.0f,
                             packed[OFF_B2 + c] * bs);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;

    if (warp == TC_COMPUTE / 32) {
        // ------------------------------------------------------------------ control lane: MMA issue
        if (tid == TC_COMPUTE) {
            int sb = 0, bphase = 0, sa = 0, aphase = 0;
#pragma unroll 1
            for (int t = 0; t < my_tiles; ++t) {
#pragma unroll 1
                for (int c = 0; c < FB_CHUNKS; ++c) {
                    mbar_wait(&a_full[sa], aphase);
                    if (c == 0 && t > 0) mbar_wait(acc_free, (t - 1) & 1);
                    if (c == 1) mbar_wait(l1_read, t & 1);               // every product starts over in the same accumulators
                    if (c == 1 + NCH) mbar_wait(l2_read, t & 1);
                    const uint32_t a_h = smem_u32(sm + OFF_A + sa * A_STAGE), a_m = a_h + A_WORD, a_l = a_m + A_WORD;
                    const bool first = (c == 0 || c == 1 || c == 1 + NCH);
#pragma unroll
                    for (int ks = 0; ks < NSUB; ++ks) {
                        mbar_wait(&b_full[sb], bphase);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t b_h = smem_u32(sm + OFF_B + sb * B_STAGE), b_m = b_h + B_WORD, b_l = b_m + B_WORD;
                        const uint32_t o = ks * 32;
                        const uint32_t acc = (first && ks == 0) ? 0u : 1u;
                        umma_bf16(tmem_d + HID, umma_desc_a(a_m + o), umma_desc_b(b_m), acc);
                        umma_bf16(tmem_d + HID, umma_desc_a(a_h + o), umma_desc_b(b_l), 1u);
                        umma_bf16(tmem_d + HID, umma_desc_a(a_l + o), umma_desc_b(b_h), 1u);
                        umma_bf16(tmem_d + HID, umma_desc_a(a_h + o), umma_desc_b(b_m), 1u);
                        umma_bf16(tmem_d + HID, umma_desc_a(a_m + o), umma_desc_b(b_h), 1u);
                        umma_bf16(tmem_d, umma_desc_a(a_h + o), umma_desc_b(b_h), acc);
                        umma_commit(&b_empty[sb]);
                        if (ks == NSUB - 1) {
                            umma_commit(&a_empty[sa]);
                            if (c == 0) umma_commit(l1_full);
                            if (c == NCH) umma_commit(l2_full);
                            if (c == FB_CHUNKS - 1) umma_commit(l3_full);
                        }
                        if (++sb == FNSB) { sb = 0; bphase ^= 1; }
                    }
                    if (++sa == FNSA) { sa = 0; aphase ^= 1; }
                }
            }
        }
    } else if (warp == TC_COMPUTE / 32 + 1) {
        // ------------------------------------------------------------------ weight stream
        if (tid == TC_COMPUTE + 32) {
            asm volatile("griddepcontrol.wait;" ::: "memory");           // the image's pack kernel (launched just before) is complete
            int sb = 0, bphase = 0, pq = 0;
#pragma unroll 1
            for (int t = 0; t < my_tiles; ++t) {
#pragma unroll 1
                for (int idx = 0; idx < FB_SUBS; ++idx, ++pq) {
                    if (pq >= FNSB) mbar_wait(&b_empty[sb], bphase ^ 1);
                    mbar_expect_tx(&b_full[sb], B_STAGE);
                    bulk_g2s(sm + OFF_B + sb * B_STAGE, image + (size_t)idx * B_STAGE, B_STAGE, &b_full[sb]);
                    if (++sb == FNSB) { sb = 0; bphase ^= 1; }
                }
            }
        }
    } else {
        // ------------------------------------------------------------------ rows
        const int r = tid & (TM - 1), part = tid >> 7, lane = tid & 31;
        const uint32_t a_off = sw64((uint32_t)r, (uint32_t)part);
        const uint32_t lane_base = tmem_d + ((uint32_t)((warp & 3) * 32) << 16);
        constexpr int CPT = HID / NPART;                                // 64 columns per thread
        const float sc = TANH ? kTwoLog2e : 1.0f;
        int sa = 0, aphase = 0, qa = 0;
        auto tile_row0 = [&](int tt) { return ((int64_t)blockIdx.x + (int64_t)tt * gridDim.x) * TM; };
        // writes this thread's 16 bytes of the three word buffers of the next ring stage and hands the stage over
        auto push_chunk = [&](const float (&v)[UPT]) {
            uint4 H, M, L;
            split8(v, H, M, L);
            if (qa >= FNSA) mbar_wait(&a_empty[sa], aphase ^ 1);
            unsigned char* a0 = sm + OFF_A + sa * A_STAGE + a_off;
            *reinterpret_cast<uint4*>(a0) = H;
            *reinterpret_cast<uint4*>(a0 + A_WORD) = M;
            *reinterpret_cast<uint4*>(a0 + 2 * A_WORD) = L;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            warp_arrive(&a_full[sa]);
            ++qa;
            if (++sa == FNSA) { sa = 0; aphase ^= 1; }
        };
        // gathers the minibatch rows (ppo_continuous.py:217 s[index]): the layer-1 operand and the padded copy for dW1
        // source row of minibatch row `row` (ppo_continuous.py:217 index), fetched a phase ahead of its uses
        auto src_of = [&](int64_t row) { return row < n ? (index ? index[row] : row) : (int64_t)0; };
        auto produce_x = [&](int tt, int64_t src) {
            const int64_t row = tile_row0(tt) + r;
            const bool live = row < n;
            const int k0 = part * UPT;
            float v[UPT], xv[UPT];
#pragma unroll
            for (int j = 0; j < UPT; ++j) v[j] = s[src * IN + (k0 + j < IN ? k0 + j : 0)];
#pragma unroll
            for (int j = 0; j < UPT; ++j) xv[j] = (live && k0 + j < IN) ? v[j] : 0.0f;
            push_chunk(xv);
            float4* xo = reinterpret_cast<float4*>(xs + row * XS_LD + k0);
            xo[0] = make_float4(xv[0], xv[1], xv[2], xv[3]);
            xo[1] = make_float4(xv[4], xv[5], xv[6], xv[7]);
        };
        produce_x(0, src_of(tile_row0(0) + r));
#pragma unroll 1
        for (int t = 0; t < my_tiles; ++t) {
            const int tile = (int)blockIdx.x + t * (int)gridDim.x;
            const int64_t row = tile_row0(t) + r;
            const bool live = row < n;
            const int64_t wrow0 = row - lane;                            // first row of this warp's 32 rows
            const int64_t src = src_of(row);                             // used by the loss phase
            const int64_t src_next = (t + 1 < my_tiles) ? src_of(tile_row0(t + 1) + r) : 0;
            float* st = stg + warp * ST_WARP;
            float va[CPT];                                               // pre1 -> h1, then acc2 -> h2 -> dz2, then dh1
            // ---------------- layer 1: h1 = act(W1 x + b1), eight operand chunks, h1 to HBM
            FB_TRACE(t * 16 + 0);
            mbar_wait(l1_full, t & 1);
            FB_TRACE(t * 16 + 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tmem_sum64(lane_base, part * CPT, va);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            warp_arrive(l1_read);
#pragma unroll
            for (int kc = 0; kc < NCH; ++kc) {
                float h[UPT];
#pragma unroll
                for (int j = 0; j < UPT; j += 2) {
                    const float2 bb = *reinterpret_cast<const float2*>(b1p + part * CPT + kc * UPT + j);
                    const float2 hh = act2_scaled<TANH>(__ffma2_rn(make_float2(va[kc * UPT + j], va[kc * UPT + j + 1]), make_float2(sc, sc), bb));
                    h[j] = hh.x; h[j + 1] = hh.y;
                    va[kc * UPT + j] = hh.x; va[kc * UPT + j + 1] = hh.y;
                }
                push_chunk(h);
                // h1 row-major [mp][256] (value kc * 8 + j of this thread is unit 32 kc + 8 part + j): two chunks = one batch of
                // two 32-byte segments per row, stored while the ring waits for the tensor core
                if (kc & 1)
                    store_rows_batch(kc >> 1, h1g + wrow0 * HID, HID, va, st, lane, [&](int b, int pc) { return (2 * b + (pc >> 1)) * KC + part * UPT + (pc & 1) * 4; });
            }
            FB_TRACE(t * 16 + 2);
            FB_TRACE(t * 16 + 3);
            // ---------------- layer 2: h2 = act(W2 h1 + b2) (columns 64 part .. + 63), head pre-activations
            mbar_wait(l2_full, t & 1);
            FB_TRACE(t * 16 + 4);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tmem_sum64(lane_base, part * CPT, va);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            warp_arrive(l2_read);
            // the loss phase's per-row inputs (quarter 0 only), in flight during the head sums
            float la[3] = {0.0f, 0.0f, 0.0f}, lo[3] = {0.0f, 0.0f, 0.0f}, ladv = 0.0f;
            if (part == 0 && live) {
                if (CRITIC) ladv = v_target[src];
                else {
#pragma unroll
                    for (int k = 0; k < 3; ++k) { la[k] = a[src * 3 + k]; lo[k] = old_logp[src * 3 + k]; }
                    ladv = adv[src];
                }
            }
            {
                float2 p0 = make_float2(0.0f, 0.0f), p1 = p0, p2 = p0;
#pragma unroll
                for (int j = 0; j < CPT; j += 2) {
                    const float4 wa = w3t[part * CPT + j], wb = w3t[part * CPT + j + 1];
                    const float2 h2 = act2_scaled<TANH>(__ffma2_rn(make_float2(va[j], va[j + 1]), make_float2(sc, sc), make_float2(wa.w, wb.w)));
                    va[j] = h2.x; va[j + 1] = h2.y;
                    p0 = __ffma2_rn(h2, make_float2(wa.x, wb.x), p0);
                    if (heads > 1) { p1 = __ffma2_rn(h2, make_float2(wa.y, wb.y), p1); p2 = __ffma2_rn(h2, make_float2(wa.z, wb.z), p2); }
                }
                red[part * TM + r] = make_float4(p0.x + p0.y, p1.x + p1.y, p2.x + p2.y, 0.0f);
            }
            asm volatile("bar.sync 1, %0;" ::"n"(TC_COMPUTE) : "memory");
            FB_TRACE(t * 16 + 5);
            // ---------------- per-row loss and its gradient w.r.t. the head pre-activations (quarter 0: one thread per row)
            if (part == 0) {
                float pre[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float* q = reinterpret_cast<const float*>(red) + k;
                    pre[k] = ((q[(0 * TM + r) * 4] + q[(1 * TM + r) * 4]) + q[(2 * TM + r) * 4]) + q[(3 * TM + r) * 4];
                }
                float d3[3] = {0.0f, 0.0f, 0.0f}, dls[3] = {0.0f, 0.0f, 0.0f}, loss = 0.0f;
                [[maybe_unused]] float stat[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                if (live) {
                    if (CRITIC) {
                        const float v = pre[0] + __ldg(packed + OFF_B3);
                        const float diff = v - ladv;
                        loss = diff * diff * inv_n;                                                    // :233
                        d3[0] = 2.0f * diff * inv_n;
                    } else {
                        float mean[3], sd[3], x[3], th[3], lsum = 0.0f, ent = 0.0f;
#pragma unroll
                        for (int k = 0; k < 3; ++k) {
                            th[k] = tanhf(pre[k] + __ldg(packed + OFF_B3 + k));
                            mean[k] = max_action * th[k];
                            const float ls = __ldg(packed + OFF_LS + k);
                            sd[k] = expf(ls);
                            x[k] = la[k];
                            const float diff = x[k] - mean[k];
                            lsum += -(diff * diff) / (2.0f * sd[k] * sd[k]) - ls - 0.9189385332046727f - lo[k];   // :219-221
                            ent += 1.4189385332046727f + ls;                                           // :218 Normal.entropy()
                        }
                        const float ratio = expf(lsum);
                        const float A = ladv;
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
                dz3s[r] = make_float4(d3[0], d3[1], d3[2], 0.0f);
                float rs[8] = {d3[0], d3[1], d3[2], dls[0], dls[1], dls[2], loss, 0.0f};
                if (CRITIC) { rs[1] = loss; rs[6] = 0.0f; }
#pragma unroll
                for (int k = 0; k < 7; ++k)
#pragma unroll
                    for (int off = 16; off; off >>= 1) rs[k] += __shfl_xor_sync(0xffffffffu, rs[k], off);
                if (lane == 0)
#pragma unroll
                    for (int k = 0; k < 8; ++k) scal[warp * 8 + k] = rs[k];
                if constexpr (STATS) {
                    float* statw = reinterpret_cast<float*>(sm + OFF_STAT);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
#pragma unroll
                        for (int off = 16; off; off >>= 1) stat[k] += __shfl_xor_sync(0xffffffffu, stat[k], off);
                    if (lane == 0)
#pragma unroll
                        for (int k = 0; k < 4; ++k) statw[warp * 4 + k] = stat[k];
                }
            }
            asm volatile("bar.sync 1, %0;" ::"n"(TC_COMPUTE) : "memory");
            FB_TRACE(t * 16 + 6);
            if (tid < 8) part_scal[(int64_t)tile * 8 + tid] = ((scal[tid] + scal[8 + tid]) + scal[16 + tid]) + scal[24 + tid];
            if constexpr (STATS) {
                const float* statw = reinterpret_cast<const float*>(sm + OFF_STAT);
                if (tid >= 8 && tid < 12) {
                    const int k = tid - 8;
                    part_stat[(int64_t)tile * 8 + k] = ((statw[k] + statw[4 + k]) + statw[8 + k]) + statw[12 + k];
                }
            }
            // ---------------- dz2 = (dz3 W3) act'(h2): eight operand chunks of the backward product (K order permuted), the
            // per-tile column sums of dW3 = dz3^T h2 and db2 = sum dz2, dz2 to HBM
            {
                const float4 d3 = dz3s[r];
                float* cw = colp + warp * (4 * 64);
#pragma unroll
                for (int kc = 0; kc < NCH; ++kc) {
                    float dz[UPT], qa_[16], qb_[16];
#pragma unroll
                    for (int j = 0; j < UPT; ++j) {
                        const float4 w = w3t[part * CPT + kc * UPT + j];
                        const float hv = va[kc * UPT + j];
                        float dh = d3.x * w.x;
                        if (heads > 1) dh = fmaf(d3.z, w.z, fmaf(d3.y, w.y, dh));
                        dz[j] = dh * act_grad_of<TANH>(hv);
                        va[kc * UPT + j] = dz[j];
                        qa_[j] = hv * d3.x; qa_[8 + j] = dz[j];          // quantities 0 (dW3 row 0) and 3 (db2)
                        if (heads > 1) { qb_[j] = hv * d3.y; qb_[8 + j] = hv * d3.z; }
                    }
                    push_chunk(dz);
                    warp_transpose_sum16(qa_, lane);
                    if (!(lane & 1)) cw[((lane >> 4) ? 3 : 0) * 64 + kc * UPT + ((lane >> 1) & 7)] = qa_[0];
                    if (heads > 1) {
                        warp_transpose_sum16(qb_, lane);
                        if (!(lane & 1)) cw[(1 + (lane >> 4)) * 64 + kc * UPT + ((lane >> 1) & 7)] = qb_[0];
                    }
                    // dz2 in column blocks [4][mp][64]: this thread's 64 columns are block `part`
                    if (kc & 1)
                        store_rows_batch(kc >> 1, dz2b + ((int64_t)part * mp + wrow0) * 64, 64, va, st, lane, [&](int b, int pc) { return b * 16 + pc * 4; });
                }
                FB_TRACE(t * 16 + 7);
            }
            FB_TRACE(t * 16 + 8);
            if (t + 1 < my_tiles) produce_x(t + 1, src_next);
            FB_TRACE(t * 16 + 9);                      // into the ring behind this tile's last chunk
            asm volatile("bar.sync 1, %0;" ::"n"(TC_COMPUTE) : "memory");
            {
                // the four row groups of every quarter, in a fixed order: rows 0..heads-1 = dW3, row 3 = db2
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int v = r + TM * e, q = v >> 6, cc = v & 63;
                    if (q < heads || q == 3) {
                        const float* c0 = colp + (part * 4) * (4 * 64) + q * 64 + cc;
                        part_head[((int64_t)tile * 4 + q) * HID + part * CPT + cc] = ((c0[0] + c0[4 * 64]) + c0[2 * 4 * 64]) + c0[3 * 4 * 64];
                    }
                }
            }
            // ---------------- dz1 = (dz2 W2) act'(h1) -> HBM row-major (columns 64 part .. + 63 = input units)
            FB_TRACE(t * 16 + 10);
            mbar_wait(l3_full, t & 1);
            FB_TRACE(t * 16 + 11);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tmem_sum64(lane_base, part * CPT, va);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            warp_arrive(acc_free);
            {
                auto seg = [&](int b, int pc) { return part * CPT + b * 16 + pc * 4; };
                scale_by_act_grad<TANH>(h1g + wrow0 * HID, HID, va, st, lane, seg);
                store_rows(dz1g + wrow0 * HID, HID, va, st, lane, seg);
            }
            FB_TRACE(t * 16 + 12);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == TC_COMPUTE / 32) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(kTmemCols) : "memory");
    }
}

template <typename K>
int set_smem(K kernel, int bytes) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    return e == cudaSuccess ? SAT_OK : (int)e;
}

}  // namespace

#ifdef SAT_TC_TRACE
extern "C" int sat_debug_fb_tc_trace(unsigned long long* out) { return (int)cudaMemcpyFromSymbol(out, g_fb_trace, sizeof(g_fb_trace)); }
#endif

int ppo_fb_tc_launch(bool critic, bool use_tanh, const float* packed, unsigned char* image, float max_action, const float* s,
                     const float* a, const float* old_logp, const float* adv, const float* v_target, const int64_t* index,
                     int64_t n, float inv_n, float epsilon, float entropy_coef, float* h1g, float* dz2b, float* dz1g, float* xs,
                     float* part_head, float* part_scal, int64_t mp, float* part_stat, cudaStream_t stream) {
    if (mp % TM) return SAT_ERR_SIZE;
    if (part_stat && critic) return SAT_ERR_SIZE;
    static int sm_count[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    int sms = (dev >= 0 && dev < 64) ? sm_count[dev] : 0;
    if (sms <= 0) {
        e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 0 && dev < 64) sm_count[dev] = sms;
    }
    // the image is rebuilt from the packed weights on every call: the Adam kernel rewrites them after every minibatch
    ppo_fb_tc_pack_kernel<<<(FB_CHUNKS * 4 * HID + 255) / 256, 256, 0, stream>>>(packed, image);
    const int64_t tiles = mp / TM;
    const unsigned blocks = (unsigned)(tiles < sms ? tiles : sms);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = FB_SMEM; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;     // overlap the kernel's prologue with the pack kernel
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
#define SAT_FB_LAUNCH(C, T, S)                                                                                                 \
    do {                                                                                                                       \
        cfg.dynamicSmemBytes = S ? FB_SMEM_STATS : FB_SMEM;                                                                    \
        int rc = set_smem(ppo_fb_tc_kernel<C, T, S>, (int)cfg.dynamicSmemBytes);                                              \
        if (rc) return rc;                                                                                                     \
        e = cudaLaunchKernelEx(&cfg, ppo_fb_tc_kernel<C, T, S>, packed, (const unsigned char*)image, max_action, s, a, old_logp, adv, v_target, \
                               index, n, inv_n, epsilon, entropy_coef, h1g, dz2b, dz1g, xs, part_head, part_scal, mp, part_stat); \
        if (e != cudaSuccess) return (int)e;                                                                                   \
    } while (0)
    if (critic) { if (use_tanh) SAT_FB_LAUNCH(true, true, false); else SAT_FB_LAUNCH(true, false, false); }
    else if (part_stat) { if (use_tanh) SAT_FB_LAUNCH(false, true, true); else SAT_FB_LAUNCH(false, false, true); }
    else { if (use_tanh) SAT_FB_LAUNCH(false, true, false); else SAT_FB_LAUNCH(false, false, false); }
#undef SAT_FB_LAUNCH
    e = cudaGetLastError();
    return e == cudaSuccess ? SAT_OK : (int)e;
}
