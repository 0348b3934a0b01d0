// actor_tc.cu -- K3 on the 5th-generation tensor cores: both dense layers of Actor_Gaussian (18 -> 256 -> 256) as
// error-free-split BF16x3 products on tcgen05.mma with the accumulators in TMEM (sm_100a only).
//
// Reference behaviour replaced: the same as actor.cu (PPO_continuous.choose_action -> Actor_Gaussian.forward,
// ppo_continuous.py:83-95, 176-189), which the reference evaluates in fp32.
//
// Why: config 3 "with fused actor sampling" spends 67 % of its step in the two FFMA2 actor launches (2 x 193 us at
// 65 536 rows, 65 % of the nominal fp32 rate: the CUDA-core ceiling). The hidden layer is a 65 536 x 256 x 256
// contraction. A plain bf16 / TF32 product would be narrower than the reference's fp32, so every fp32 operand is split
// EXACTLY into three bf16 words (x = h + m + l, 8 significant bits each, by truncation) and six of the nine word
// products are accumulated in fp32 in TMEM:
//     A B ~= A_h B_h  +  (A_h B_m + A_m B_h)  +  (A_m B_m + A_h B_l + A_l B_h)        (dropped: ~2^-24 relative).
// Round 2's first version used two TF32 words (3xTF32): its error against an fp64 ground truth was 1.6x the FFMA2
// kernel's, because the tensor core's fp32 accumulation TRUNCATES and every 22-bit TF32 x TF32 product loses bits when
// it is added to a larger accumulator (32 such additions per output). A bf16 x bf16 product has 16 significant bits,
// so the large A_h B_h term is added (nearly always) exactly, in 16 instead of 32 accumulations (UMMA K = 16), and all
// the rounding happens in the SECOND accumulator, whose content is 2^-8 of the result. Same number of MMA instructions
// (6 products x 2 k-steps per 32-unit chunk instead of 3 x 4) and 25 % fewer operand bytes (6 instead of 8 per value).
// tests/test_gpu_actor_tc.py measures the error of this path and of the FFMA2 path against an fp64 ground truth.
//
// Persistent kernel, one CTA per SM; a row tile = 128 observations (= the 128 TMEM lanes), 544 threads:
//   warps 0-15 (thread = row r = tid & 127, quarter p = tid >> 7):
//             chunk 0: rebuild / load 8 of the row's observation values, split, write the layer-1 A operand (K = 18
//             padded to 32); when the layer-1 MMAs are complete, tcgen05.ld 64 pre-activations (the W1 image permutes
//             the output units so that a thread's 64 units - 8 per later chunk - are 64 CONSECUTIVE accumulator columns);
//             chunks 1..8: bias, tanh, split, the K-major 64-byte-swizzled A operand of 32 hidden units;
//             epilogue: tcgen05.ld of 64 of the row's accumulator columns (a warp may only touch TMEM lanes
//             32 (w % 4) .. +31, which is exactly its rows), bias, tanh, partial head dot products, reduced over the four
//             quarters through shared memory; thread (r, p < 3) then finishes action p: Philox sample, clamp, log-prob;
//   warp 16, one elected lane: streams the pre-split, pre-swizzled weight image (48 KB per chunk: W1 then the eight
//             K-chunks of W2, h | m | l) through a three-stage shared-memory ring with cp.async.bulk + mbarrier and issues
//             the 12 tcgen05.mma (kind::f16, M 128, N 256, K 16) of each chunk; tcgen05.commit hands the stages back and
//             signals "layer 1 complete" / "layer 2 complete".
// TMEM: columns [0, 256) A_h B_h, [256, 512) the five small products; layer 1 uses the same columns before layer 2.
// Across tiles: the weight ring never drains, the next tile's observation operand is written while the current tile's last
// chunks are on the tensor core, and its layer-1 MMAs start as soon as the epilogue has the accumulators in registers.
// Shared memory: A 2 x 24 KB, X 24 KB, B 3 x 48 KB, head table 4 KB, bias 1 KB = 222 KB -> one CTA per SM.
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>
#include "sat_math.cuh"
#include "tc_mlp.cuh"

namespace {
using namespace mlp;
using namespace tcm;

constexpr int OFF_A = 0;                        // A ring: FIFO over the observation operand and the eight hidden chunks of every tile
constexpr int OFF_B = OFF_A + NSA * A_STAGE;
constexpr int OFF_RED = OFF_B + NSB * B_STAGE;  // head partial sums [2 tiles][NPART][TM] float4
constexpr int OFF_W3P = OFF_RED + 2 * NPART * TM * 16;  // per column pair (a, b) two float4: (b2a', b2b', w0a, w0b), (w1a, w1b, w2a, w2b)
constexpr int OFF_B1P = OFF_W3P + 2 * HID * 16; // b1 in layer-1 accumulator column order (both tables: one per network)
constexpr int OFF_BAR = OFF_B1P + 2 * HID * 4;  // mbarriers
constexpr int OFF_TMEM = OFF_BAR + 24 * 8;
constexpr int TC_SMEM = OFF_TMEM + 16 + 1024;   // + slack for the 1024-byte alignment of the swizzled tiles
static_assert(TC_SMEM <= 227 * 1024, "shared memory budget");
static_assert(NCHUNK * NSUB * B_STAGE <= SAT_ACTOR_TC_IMAGE_FLOATS * 4, "weight image larger than the caller's scratch");

// The weight image: chunk 0 = W1 (n = layer-1 accumulator column, k = observation dimension, zero beyond 18), chunks 1..8 =
// the K-chunks of W2 (n = output unit); every chunk is two sub-chunks of 16 k (one UMMA k-step), each [h | m | l] x 256 rows x
// 32 bytes, 8-row groups of 256 bytes with the two 16-byte halves XOR-swizzled: exactly the bytes the SWIZZLE_32B descriptor
// expects, so one linear 24 KB bulk copy per sub-chunk brings it in. packed: the FFMA kernel's image (W1T[k][j],
// W2T[k][n] = fc2.weight[n][k]). One thread = 8 consecutive k of one n (coalesced over n).
__global__ void actor_tc_pack_kernel(const float* __restrict__ packed0, unsigned char* __restrict__ image0,
                                     const float* __restrict__ packed1, unsigned char* __restrict__ image1) {
    // programmatic dependent launch: the sampling kernel may start its prologue (barriers, TMEM, tables, first observation
    // operand) now; its weight-stream lane waits for this grid to complete before it reads the image
    asm volatile("griddepcontrol.launch_dependents;");
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= NCHUNK * 4 * HID) return;
    const float* __restrict__ packed = blockIdx.y ? packed1 : packed0;
    unsigned char* __restrict__ image = blockIdx.y ? image1 : image0;
    const int n = idx % HID, c16 = (idx / HID) & 3, chunk = idx / (4 * HID);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int kk = c16 * 8 + j;
        if (chunk == 0) v[j] = (kk < IN) ? packed[OFF_W1T + kk * HID + l1_unit(n)] : 0.0f;
        else v[j] = packed[OFF_W2T + ((chunk - 1) * KC + kk) * HID + n];
    }
    uint4 H, M, L;
    split8(v, H, M, L);
    unsigned char* base = image + (size_t)(chunk * NSUB + (c16 >> 1)) * B_STAGE + sw32((uint32_t)n, (uint32_t)(c16 & 1));
    *reinterpret_cast<uint4*>(base) = H;
    *reinterpret_cast<uint4*>(base + B_WORD) = M;
    *reinterpret_cast<uint4*>(base + 2 * B_WORD) = L;
}

// A frozen snapshot's bias / head tables in global memory, in exactly the layout of the kernel's shared-memory tables (one
// network): w3p[HID] float4 (per column pair (b2a', b2b', w0a, w0b), (w1a, w1b, w2a, w2b)), then b1p[HID] in layer-1
// accumulator column order; tanh networks carry b1 and b2 pre-multiplied by 2 log2(e) like the kernel's own tables.
constexpr int TAB_W3P = 0, TAB_B1P = 4 * HID;
static_assert(TAB_B1P + HID == SAT_ACTOR_TC_TABLE_FLOATS, "header constant out of sync");
__global__ void actor_tc_table_kernel(const float* __restrict__ pk, float* __restrict__ tables, int use_tanh) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= HID) return;
    const float bs = use_tanh ? kTwoLog2e : 1.0f;
    tables[TAB_B1P + c] = pk[OFF_B1 + l1_unit(c)] * bs;
    const int pr = c >> 1, hb = c & 1;
    float* q0 = tables + TAB_W3P + 8 * pr;
    q0[hb] = pk[OFF_B2 + c] * bs;
    q0[2 + hb] = pk[OFF_W3 + c];
    q0[4 + hb] = pk[OFF_W3 + HID + c];
    q0[6 + hb] = pk[OFF_W3 + 2 * HID + c];
}

// the opponent groups of a pool launch (kernel parameter space): group k covers rows [row_end[k - 1], row_end[k])
struct TcPool {
    const float* packed[SAT_ACTOR_POOL_MAX_GROUPS];
    const unsigned char* image[SAT_ACTOR_POOL_MAX_GROUPS];
    const float* tables[SAT_ACTOR_POOL_MAX_GROUPS];
    int64_t row_end[SAT_ACTOR_POOL_MAX_GROUPS];
    float max_action[SAT_ACTOR_POOL_MAX_GROUPS];
    int groups;
};
struct TcNoPool {};
// the group holding row row0 (a row tile never straddles two groups: every interior bound is a multiple of TM)
__device__ __forceinline__ int pool_group(const TcPool& p, int64_t row0) {
    int k = 0;
    while (k + 1 < p.groups && row0 >= p.row_end[k]) ++k;
    return k;
}

#ifdef SAT_TC_TRACE
// tuning aid (never compiled into the shipped library): CTA 0 records %globaltimer at pipeline events
__device__ unsigned long long g_tc_trace[2][256];
__device__ __forceinline__ void tc_trace(int who, int slot) {
    if (blockIdx.x == 0 && slot < 256) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); g_tc_trace[who][slot] = t; }
}
#define TC_TRACE(who, slot) tc_trace(who, slot)
#else
#define TC_TRACE(who, slot)
#endif

// the row's observation dimensions [8 part, 8 part + 8), split into the layer-1 A operand (one 16-byte chunk of each word buffer)
__device__ __forceinline__ void produce_x(unsigned char* xs, uint32_t a_off, int part, int64_t g, bool live,
                                          const float* __restrict__ obs_f32, const SatEnvState& st,
                                          const double* __restrict__ obs_stats, float (&xv)[UPT]) {
    // all loads are issued before anything is computed (indices clamped instead of branching: the eight values' memory
    // latencies overlap; with a branch per value they were paid one after the other, 7 us per tile on the state path)
    const int k0 = part * UPT;
    if (obs_f32) {
        float v[UPT];
#pragma unroll
        for (int j = 0; j < UPT; ++j) v[j] = obs_f32[g * IN + (k0 + j < IN ? k0 + j : 0)];
#pragma unroll
        for (int j = 0; j < UPT; ++j) xv[j] = (k0 + j < IN) ? v[j] : 0.0f;
    } else {
        // rebuild the observation from the fp64 SoA env state (environment.py:76-77: P - E, Pv - Ev, P, Pv, E, Ev), normalise in
        // fp64 (normalization.py:41); columns: k < 6 -> state[k] - state[k + 6], else state[k - 6]
        const int64_t ld = st.ld;
#pragma unroll
        for (int h = 0; h < UPT; h += 4) {
            double ya[4], yb[4], mu[4], sd[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = (k0 + h + j < IN) ? k0 + h + j : 0;
                ya[j] = st.state[(k < 6 ? k : k - 6) * ld + g];
                yb[j] = st.state[(k < 6 ? k + 6 : k - 6) * ld + g];
                mu[j] = obs_stats ? obs_stats[1 + k] : 0.0;
                sd[j] = obs_stats ? obs_stats[1 + 2 * IN + k] : 0.0;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = k0 + h + j;
                double y = (k < 6) ? ya[j] - yb[j] : ya[j];
                if (obs_stats) y = (y - mu[j]) / (sd[j] + 1e-8);
                xv[h + j] = (k < IN) ? (float)y : 0.0f;
            }
        }
    }
    uint4 H, M, L;
    split8(xv, H, M, L);
    unsigned char* a0 = xs + a_off;
    *reinterpret_cast<uint4*>(a0) = H;
    *reinterpret_cast<uint4*>(a0 + A_WORD) = M;
    *reinterpret_cast<uint4*>(a0 + 2 * A_WORD) = L;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // generic-proxy stores -> visible to the tensor core
}
// the fp32 observation actually fed to the network, written AFTER the operand hand-off: the proxy fence in produce_x is a
// MEMBAR that would otherwise wait for these global stores
__device__ __forceinline__ void store_obs(float* __restrict__ obs_out, int part, int64_t g, const float (&xv)[UPT]) {
#pragma unroll
    for (int j = 0; j < UPT; ++j)
        if (part * UPT + j < IN) obs_out[g * IN + part * UPT + j] = xv[j];
}
// L2 prefetch of what produce_x will read for row g (issued a tile ahead)
__device__ __forceinline__ void prefetch_x(int part, int64_t g, int64_t n, const float* __restrict__ obs_f32, const SatEnvState& st) {
    if (g >= n || part * UPT >= IN) return;
    if (obs_f32) asm volatile("prefetch.global.L2 [%0];" ::"l"(obs_f32 + g * IN + part * UPT));
    else {
#pragma unroll
        for (int j = 0; j < UPT; ++j) {
            const int k = part * UPT + j;
            if (k < IN) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(st.state + (k < 6 ? k : k - 6) * st.ld + g));
                if (k < 6) asm volatile("prefetch.global.L2 [%0];" ::"l"(st.state + (k + 6) * st.ld + g));
            }
        }
    }
}
// Persistent: one CTA per SM walks over row tiles blockIdx.x, blockIdx.x + gridDim.x, ... The weight sub-chunks stream through
// the B ring continuously across tiles; the A ring is a FIFO over (observation operand, 8 hidden chunks) of successive tiles,
// four stages deep, so the rows run up to four chunks ahead of the tensor core and the hand-off latency (stores, proxy fence,
// mbarrier, MMA issue) is hidden; the next tile's observation operand is produced while the last hidden-layer MMAs of the
// current tile run, and its layer-1 MMAs start as soon as the epilogue has the accumulators in registers.
// one network of a launch: the pursuer's and the evader's actor of a rollout step (CPPO_main.py:122-123) run in ONE persistent
// grid on the same observations (2 x ntiles tiles over the SMs instead of two launches with their own tails)
struct TcNet {
    const float* packed;
    const unsigned char* image;
    const float* eps_in;
    float *act, *logp, *mean_out, *eps_out;
    uint64_t step;
    float max_action;
};

// POOL: network 1 is an opponent pool (nnet = 2, net1 holds only the outputs and the step): an opponent tile streams the
// image of the group holding its rows, reads that group's bias / head tables from global memory (the shared-memory tables
// hold network 0's only) and its b3 / log_std / max_action from the group; the learner's tiles are network 0's as above.
template <bool TANH, bool POOL>
__global__ void __launch_bounds__(TC_THREADS, 1)
actor_tc_kernel(const __grid_constant__ TcNet net0, const __grid_constant__ TcNet net1, const int nnet,
                const float* __restrict__ obs_f32, const SatEnvState st, const double* __restrict__ obs_stats, int64_t n,
                int64_t row_offset, uint64_t seed, float* __restrict__ obs_out,
                const __grid_constant__ std::conditional_t<POOL, TcPool, TcNoPool> pool) {
    extern __shared__ unsigned char smem_dyn[];
    // 1024-byte alignment for the swizzled tiles by pointer arithmetic on the shared array (an integer round trip would turn
    // every access into a generic-space LD/ST)
    unsigned char* sm = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    float4* w3p = reinterpret_cast<float4*>(sm + OFF_W3P);
    float* b1p = reinterpret_cast<float*>(sm + OFF_B1P);
    float* red = reinterpret_cast<float*>(sm + OFF_RED);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + OFF_BAR);
    uint64_t* b_full = bars;                  // [NSB] bulk copy of a weight sub-chunk landed
    uint64_t* b_empty = bars + NSB;           // [NSB] the sub-chunk's MMAs have read the B stage
    uint64_t* a_full = bars + 2 * NSB;        // [NSA] 128 rows of the A chunk written
    uint64_t* a_empty = a_full + NSA;         // [NSA] the chunk's MMAs have read the A stage
    uint64_t* l1_full = a_empty + NSA;        // layer-1 accumulators complete
    uint64_t* l1_read = l1_full + 1;          // every row has its layer-1 pre-activations in registers: the accumulators may be overwritten
    uint64_t* l2_full = l1_full + 2;          // layer-2 accumulators complete
    uint64_t* acc_free = l1_full + 3;         // the epilogue has read the accumulators: the next tile's layer 1 may start
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + OFF_TMEM);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int ntiles = (int)((n + TM - 1) / TM);                 // row tiles; work item u = net * ntiles + row tile
    const int my_tiles = (ntiles * nnet - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // >= 1: gridDim.x <= ntiles * nnet

    if (tid == 0) {
        for (int s = 0; s < NSB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < NSA; ++s) { mbar_init(&a_full[s], TC_COMPUTE / 32); mbar_init(&a_empty[s], 1); }
        mbar_init(l1_full, 1); mbar_init(l1_read, TC_COMPUTE / 32);
        mbar_init(l2_full, 1); mbar_init(acc_free, TC_COMPUTE / 32);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == TC_COMPUTE / 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < HID * (POOL ? 1 : nnet); i += TC_THREADS) {
        // biases pre-multiplied by 2 log2(e) for the tanh networks (the activation takes its argument in that scale)
        const int nt = i / HID, c = i % HID;
        const float* pk = nt ? net1.packed : net0.packed;
        const float bs = TANH ? kTwoLog2e : 1.0f;
        b1p[nt * HID + c] = pk[OFF_B1 + l1_unit(c)] * bs;
        const int pr = c >> 1, hb = c & 1;                                // column pair, which half
        float* q0 = reinterpret_cast<float*>(w3p + nt * HID + 2 * pr);
        q0[hb] = pk[OFF_B2 + c] * bs;
        q0[2 + hb] = pk[OFF_W3 + c];
        q0[4 + hb] = pk[OFF_W3 + HID + c];
        q0[6 + hb] = pk[OFF_W3 + 2 * HID + c];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;

    if (warp == TC_COMPUTE / 32) {
        // ------------------------------------------------------------------ control lane: MMA issue
        if (tid == TC_COMPUTE) {
            // (the weight stream is fed by warp 17, so this lane never waits for a refill and issues as far ahead as operands exist)
            int sb = 0, bphase = 0;                                      // weight sub-chunk counter pq: sb = pq % NSB, bphase = (pq / NSB) & 1
            int sa = 0, aphase = 0;                                      // A chunk counter qa = 9 t + c: sa = qa % NSA, aphase = (qa / NSA) & 1
#pragma unroll 1
            for (int t = 0; t < my_tiles; ++t) {
#pragma unroll 1
                for (int c = 0; c < NCHUNK; ++c) {
                    TC_TRACE(0, (t * NCHUNK + c) * 3);
                    mbar_wait(&a_full[sa], aphase);
                    TC_TRACE(0, (t * NCHUNK + c) * 3 + 1);
                    if (c == 0 && t > 0) mbar_wait(acc_free, (t - 1) & 1);   // the previous tile's epilogue has read its accumulators
                    if (c == 1) mbar_wait(l1_read, t & 1);                   // layer 2 starts over in the same accumulators
                    const uint32_t a_h = smem_u32(sm + OFF_A + sa * A_STAGE), a_m = a_h + A_WORD, a_l = a_m + A_WORD;
#pragma unroll
                    for (int ks = 0; ks < NSUB; ++ks) {                  // UMMA K = 16 bf16 = 32 bytes along the swizzled A row
                        mbar_wait(&b_full[sb], bphase);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t b_h = smem_u32(sm + OFF_B + sb * B_STAGE), b_m = b_h + B_WORD, b_l = b_m + B_WORD;
                        const uint32_t o = ks * 32;
                        const uint32_t acc = (c <= 1 && ks == 0) ? 0u : 1u;
                        // smallest products first into the small accumulator, the exact 16-bit products alone into the main one
                        umma_bf16(tmem_d + HID, umma_desc_a(a_m + o), umma_desc_b(b_m), acc);
                        umma_bf16(tmem_d + HID, umma_desc_a(a_h + o), umma_desc_b(b_l), 1u);
                        umma_bf16(tmem_d + HID, umma_desc_a(a_l + o), umma_desc_b(b_h), 1u);
                        umma_bf16(tmem_d + HID, umma_desc_a(a_h + o), umma_desc_b(b_m), 1u);
                        umma_bf16(tmem_d + HID, umma_desc_a(a_m + o), umma_desc_b(b_h), 1u);
                        umma_bf16(tmem_d, umma_desc_a(a_h + o), umma_desc_b(b_h), acc);
                        umma_commit(&b_empty[sb]);                       // arrives when these MMAs have read their operands
                        if (ks == NSUB - 1) {
                            umma_commit(&a_empty[sa]);
                            if (c == 0) umma_commit(l1_full);
                            if (c == NCHUNK - 1) umma_commit(l2_full);
                        }
                        if (++sb == NSB) { sb = 0; bphase ^= 1; }
                    }
                    TC_TRACE(0, (t * NCHUNK + c) * 3 + 2);
                    if (++sa == NSA) { sa = 0; aphase ^= 1; }
                }
            }
        }
    } else if (warp == TC_COMPUTE / 32 + 1) {
        // ------------------------------------------------------------------ weight stream: 24 KB sub-chunks, W1 then W2, tile after tile
        if (tid == TC_COMPUTE + 32) {
            constexpr int SUBS = NCHUNK * NSUB;                          // weight sub-chunks per tile: 18
            asm volatile("griddepcontrol.wait;" ::: "memory");           // the image's pack kernel (launched just before) is complete
            int sb = 0, bphase = 0, pq = 0;
#pragma unroll 1
            for (int t = 0; t < my_tiles; ++t) {
                const int u = (int)blockIdx.x + t * (int)gridDim.x;
                const unsigned char* img = (u >= ntiles) ? net1.image : net0.image;
                if constexpr (POOL) { if (u >= ntiles) img = pool.image[pool_group(pool, (int64_t)(u - ntiles) * TM)]; }
#pragma unroll 1
                for (int idx = 0; idx < SUBS; ++idx, ++pq) {
                    if (pq >= NSB) mbar_wait(&b_empty[sb], bphase ^ 1);  // the MMAs of sub-chunk pq - NSB have read this stage
                    mbar_expect_tx(&b_full[sb], B_STAGE);
                    bulk_g2s(sm + OFF_B + sb * B_STAGE, img + (size_t)idx * B_STAGE, B_STAGE, &b_full[sb]);
                    if (++sb == NSB) { sb = 0; bphase ^= 1; }
                }
            }
        }
    } else {
        // ------------------------------------------------------------------ rows
        const int r = tid & (TM - 1), part = tid >> 7;
        const uint32_t a_off = sw64((uint32_t)r, (uint32_t)part);       // this thread's 16 bytes of every A word buffer
        const uint32_t lane_base = tmem_d + ((uint32_t)((warp & 3) * 32) << 16);
        constexpr int CPT = HID / NPART;                                // accumulator columns per thread: 64
        const float sc = TANH ? kTwoLog2e : 1.0f;
        int sa = 0, aphase = 0, qa = 0;                                 // A chunk counter (same sequence as the control lane)
        // work item t of this CTA: network and first row (network 1's tiles follow network 0's; the fp32 observation is written
        // once, by network 0's tiles)
        auto tile_net = [&](int tt) { return ((int)blockIdx.x + tt * (int)gridDim.x >= ntiles) ? 1 : 0; };
        auto tile_row0 = [&](int tt) { const int u = (int)blockIdx.x + tt * (int)gridDim.x; return (int64_t)(u >= ntiles ? u - ntiles : u) * TM; };
        {
            int64_t g = tile_row0(0) + r;
            const bool live = g < n;
            float xv[UPT];
            produce_x(sm + OFF_A, a_off, part, live ? g : n - 1, live, obs_f32, st, obs_stats, xv);
            warp_arrive(&a_full[0]);
            if (obs_out && live && !tile_net(0)) store_obs(obs_out, part, g, xv);
            sa = 1; qa = 1;
        }
        // finishes action `part` of row r of tile tt from the four quarters' head partial sums: Philox sample, clamp, log-prob
        auto sample_tile = [&](int tt) {
            const int64_t g = tile_row0(tt) + r;
            if (g >= n || part >= 3) return;
            const int a = part;
            const TcNet& nt = tile_net(tt) ? net1 : net0;
            const float* __restrict__ packed = nt.packed;
            const float* __restrict__ eps_in = nt.eps_in;
            const uint64_t step = nt.step;
            float max_action = nt.max_action;
            if constexpr (POOL) {
                if (tile_net(tt)) { const int k = pool_group(pool, tile_row0(tt)); packed = pool.packed[k]; max_action = pool.max_action[k]; }
            }
            const float* rd = red + (tt & 1) * (NPART * TM * 4);
            const float pre_a = ((rd[(0 * TM + r) * 4 + a] + rd[(1 * TM + r) * 4 + a]) + rd[(2 * TM + r) * 4 + a]) + rd[(3 * TM + r) * 4 + a];
            float eps;
            if (eps_in) eps = eps_in[g * 3 + a];
            else {
                const uint64_t gid = (uint64_t)(row_offset + g);
                uint32_t c[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)step, (uint32_t)(step >> 32)};
                sat::philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
                // Box-Muller on (0,1) uniforms: (c0, c1) -> eps 0, 1; (c2, c3) -> eps 2 (same draws as actor.cu)
                const uint32_t ca = (a == 2) ? c[2] : c[0], cb2 = (a == 2) ? c[3] : c[1];
                const float ua = ((float)ca + 0.5f) * 2.3283064365386963e-10f, ub = ((float)cb2 + 0.5f) * 2.3283064365386963e-10f;
                const float rr = sqrtf(-2.0f * logf(fminf(ua, 0.99999994f)));
                float sn, cs;
                sincosf(6.283185307179586f * ub, &sn, &cs);
                eps = rr * ((a == 1) ? sn : cs);
            }
            const float mean = max_action * tanhf(pre_a + __ldg(packed + OFF_B3 + a));                        // :87
            const float sd = expf(__ldg(packed + OFF_LS + a));                                               // :93
            float xs = fmaf(sd, eps, mean);                                                                  // :186
            xs = fminf(fmaxf(xs, -max_action), max_action);                                                  // :187
            const float diff = xs - mean;
            const float lp = -(diff * diff) / (2.0f * sd * sd) - logf(sd) - 0.9189385332046727f;             // :188
            nt.act[g * 3 + a] = xs; nt.logp[g * 3 + a] = lp;
            if (nt.mean_out) nt.mean_out[g * 3 + a] = mean;
            if (nt.eps_out) nt.eps_out[g * 3 + a] = eps;
        };
#pragma unroll 1
        for (int t = 0; t < my_tiles; ++t) {
            int tab = tile_net(t) * HID;                                // this tile's bias / head tables
            const float* b1t = b1p;
            const float4* w3t = w3p;
            if constexpr (POOL) {
                if (tile_net(t)) {                                      // an opponent's tables: global, broadcast loads
                    const float* tg = pool.tables[pool_group(pool, tile_row0(t))];
                    b1t = tg + TAB_B1P; w3t = reinterpret_cast<const float4*>(tg + TAB_W3P); tab = 0;
                }
            }
            if (t + 1 < my_tiles) prefetch_x(part, tile_row0(t + 1) + r, n, obs_f32, st);
            // ---- layer-1 pre-activations of the thread's 64 hidden units (columns [64 part, +64) of both accumulators)
            float pre1[CPT];
            if (tid == 0) TC_TRACE(1, t * 16);
            mbar_wait(l1_full, t & 1);
            if (tid == 0) TC_TRACE(1, t * 16 + 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tmem_sum64(lane_base, part * CPT, pre1);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            warp_arrive(l1_read);
            if (tid == 0) TC_TRACE(1, t * 16 + 2);
            // ---- chunks 1..8: h1 = act(pre1 + b1), split, A operand of 32 hidden units
#pragma unroll
            for (int kc = 0; kc < NCH; ++kc) {
                // the previous tile's sampling, where the rows are a full ring ahead of the tensor core (its head partial sums
                // sit in the other half of the scratch; every thread is past its epilogue here)
                if (kc == NSA && t > 0) {
                    asm volatile("bar.sync 1, %0;" ::"n"(TC_COMPUTE) : "memory");   // the 16 compute warps only
                    sample_tile(t - 1);
                }
                float h[UPT];
#pragma unroll
                for (int j = 0; j < UPT; j += 2) {
                    const float2 bb = *reinterpret_cast<const float2*>(b1t + tab + part * CPT + kc * UPT + j);
                    const float2 hh = act2_scaled<TANH>(__ffma2_rn(make_float2(pre1[kc * UPT + j], pre1[kc * UPT + j + 1]), make_float2(sc, sc), bb));
                    h[j] = hh.x; h[j + 1] = hh.y;
                }
                uint4 H, M, L;
                split8(h, H, M, L);
                if (qa >= NSA) mbar_wait(&a_empty[sa], aphase ^ 1);     // the MMAs of A chunk qa - NSA have consumed this stage
                unsigned char* a0 = sm + OFF_A + sa * A_STAGE + a_off;
                *reinterpret_cast<uint4*>(a0) = H;
                *reinterpret_cast<uint4*>(a0 + A_WORD) = M;
                *reinterpret_cast<uint4*>(a0 + 2 * A_WORD) = L;
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                warp_arrive(&a_full[sa]);
                if (tid == 0) TC_TRACE(1, t * 16 + 3 + kc);
                ++qa;
                if (++sa == NSA) { sa = 0; aphase ^= 1; }
            }
            // ---- the next tile's observation operand goes into the ring behind this tile's last chunk
            if (t + 1 < my_tiles) {
                int64_t gn = tile_row0(t + 1) + r;
                const bool live_n = gn < n;
                if (qa >= NSA) mbar_wait(&a_empty[sa], aphase ^ 1);
                if (tid == 0) TC_TRACE(1, t * 16 + 15);
                float xv[UPT];
                produce_x(sm + OFF_A + sa * A_STAGE, a_off, part, live_n ? gn : n - 1, live_n, obs_f32, st, obs_stats, xv);
                warp_arrive(&a_full[sa]);
                if (obs_out && live_n && !tile_net(t + 1)) store_obs(obs_out, part, gn, xv);
                ++qa;
                if (++sa == NSA) { sa = 0; aphase ^= 1; }
            }

            // ------------------------------------------------------------------ epilogue: h2 = act(D + b2), head partial sums
            if (tid == 0) TC_TRACE(1, t * 16 + 11);
            mbar_wait(l2_full, t & 1);
            if (tid == 0) TC_TRACE(1, t * 16 + 12);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            float acc2[CPT];
            tmem_sum64(lane_base, part * CPT, acc2);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            warp_arrive(acc_free);                                       // accumulators are in registers: the next tile's layer 1 may run
            if (tid == 0) TC_TRACE(1, t * 16 + 13);
            float2 p0 = make_float2(0.0f, 0.0f), p1 = p0, p2 = p0;
#pragma unroll
            for (int j = 0; j < CPT; j += 2) {
                const float4 qa4 = w3t[tab + part * CPT + j], qb4 = w3t[tab + part * CPT + j + 1];   // pair (j, j + 1): two broadcast loads
                const float2 h2 = act2_scaled_fma<TANH>(__ffma2_rn(make_float2(acc2[j], acc2[j + 1]), make_float2(sc, sc), make_float2(qa4.x, qa4.y)));
                p0 = __ffma2_rn(h2, make_float2(qa4.z, qa4.w), p0);
                p1 = __ffma2_rn(h2, make_float2(qb4.x, qb4.y), p1);
                p2 = __ffma2_rn(h2, make_float2(qb4.z, qb4.w), p2);
            }
            // the four quarters of every row meet in shared memory (double-buffered over tiles: the sampling of tile t runs
            // during tile t + 1)
            *reinterpret_cast<float4*>(red + (t & 1) * (NPART * TM * 4) + (part * TM + r) * 4) = make_float4(p0.x + p0.y, p1.x + p1.y, p2.x + p2.y, 0.0f);
            if (tid == 0) TC_TRACE(1, t * 16 + 14);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(TC_COMPUTE) : "memory");
        sample_tile(my_tiles - 1);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == TC_COMPUTE / 32) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(kTmemCols) : "memory");
    }
}

inline int launch_status() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? SAT_OK : (int)e;
}

}  // namespace

#ifdef SAT_TC_TRACE
extern "C" int sat_debug_actor_tc_trace(unsigned long long* out) { return (int)cudaMemcpyFromSymbol(out, g_tc_trace, sizeof(g_tc_trace)); }
#endif

namespace {
// once per device: the kernels' shared-memory opt-in; the SM count (cached)
int tc_setup(int* sms_out) {
    static unsigned char done[64] = {0};
    static int sm_count[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    const bool cached = dev >= 0 && dev < 64;
    if (!cached || !done[dev]) {
        e = cudaFuncSetAttribute(actor_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
        if (e != cudaSuccess) return (int)e;
        e = cudaFuncSetAttribute(actor_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
        if (e != cudaSuccess) return (int)e;
        e = cudaFuncSetAttribute(actor_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
        if (e != cudaSuccess) return (int)e;
        e = cudaFuncSetAttribute(actor_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
        if (e != cudaSuccess) return (int)e;
        if (cached) done[dev] = 1;
    }
    int sms = cached ? sm_count[dev] : 0;
    if (sms <= 0) {
        e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return (int)e;
        if (cached) sm_count[dev] = sms;
    }
    *sms_out = sms;
    return SAT_OK;
}

// launches the persistent kernel for one network (b == nullptr) or two networks on the same observations
int launch_tc(const SatActorWeights* wa, float* image_a, const SatActorWeights* wb, float* image_b, const float* obs_f32,
              const SatEnvState* st, const double* obs_stats, int64_t n, int64_t row_offset, uint64_t seed, uint64_t step_a,
              uint64_t step_b, const float* eps_in, float* act_a, float* logp_a, float* mean_out, float* eps_out, float* obs_out,
              float* act_b, float* logp_b, void* stream) {
    const int nnet = wb ? 2 : 1;
    if (!wa || !wa->packed || !image_a || !act_a || !logp_a || (!obs_f32 && !st)) return SAT_ERR_NULL;
    if (wb && (!wb->packed || !image_b || !act_b || !logp_b)) return SAT_ERR_NULL;
    if (wa->in_dim != IN || wa->hidden != HID || wa->act_dim != 3) return SAT_ERR_SIZE;
    if (wb && (wb->in_dim != IN || wb->hidden != HID || wb->act_dim != 3)) return SAT_ERR_SIZE;
    if (wb && (wb->use_tanh != 0) != (wa->use_tanh != 0)) return SAT_ERR_MODE;       // one activation per launch
    if (n <= 0 || ((uintptr_t)wa->packed & 15) || ((uintptr_t)image_a & 15)) return SAT_ERR_SIZE;
    if (wb && (((uintptr_t)wb->packed & 15) || ((uintptr_t)image_b & 15))) return SAT_ERR_SIZE;
    if (!obs_f32 && (st->n < n || st->ld < st->n)) return SAT_ERR_SIZE;
    int sms = 0;
    cudaError_t e = (cudaError_t)tc_setup(&sms);
    if (e != cudaSuccess) return (int)e;
    cudaStream_t s = (cudaStream_t)stream;
    // the images are rebuilt from the live weights on every call (a few microseconds): they can never be stale
    TcNet n0 = {wa->packed, reinterpret_cast<unsigned char*>(image_a), eps_in, act_a, logp_a, mean_out, eps_out, step_a, wa->max_action};
    TcNet n1 = n0;
    if (wb) n1 = {wb->packed, reinterpret_cast<unsigned char*>(image_b), nullptr, act_b, logp_b, nullptr, nullptr, step_b, wb->max_action};
    actor_tc_pack_kernel<<<dim3((NCHUNK * 4 * HID + 255) / 256, nnet), 256, 0, s>>>(n0.packed, const_cast<unsigned char*>(n0.image),
                                                                                    n1.packed, const_cast<unsigned char*>(n1.image));
    int rc = launch_status();
    if (rc) return rc;
    SatEnvState s0 = {};
    if (!obs_f32) s0 = *st;
    const int64_t work = ((n + TM - 1) / TM) * nnet;
    const unsigned blocks = (unsigned)(work < sms ? work : sms);          // persistent: one CTA per SM walks over the tiles
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = TC_SMEM; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;     // overlap this kernel's prologue with the pack kernel
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    e = wa->use_tanh ? cudaLaunchKernelEx(&cfg, actor_tc_kernel<true, false>, n0, n1, nnet, obs_f32, s0, obs_stats, n, row_offset, seed, obs_out, TcNoPool{})
                     : cudaLaunchKernelEx(&cfg, actor_tc_kernel<false, false>, n0, n1, nnet, obs_f32, s0, obs_stats, n, row_offset, seed, obs_out, TcNoPool{});
    return e == cudaSuccess ? launch_status() : (int)e;
}

// the learner on all rows and the snapshot of every group on its rows, in one persistent grid: the learner's image is rebuilt
// from its live weights (the snapshots' images are frozen, built once by sat_actor_tc_snapshot)
int launch_pool(const SatActorWeights* wa, float* image_a, const SatActorPoolGroup* groups, int ngroups, const float* obs_f32,
                const SatEnvState* st, const double* obs_stats, int64_t n, int64_t row_offset, uint64_t seed, uint64_t step_a,
                uint64_t step_b, float* act_a, float* logp_a, float* obs_out, float* act_b, float* logp_b, void* stream) {
    if (!wa || !wa->packed || !image_a || !groups || !act_a || !logp_a || !act_b || !logp_b || (!obs_f32 && !st)) return SAT_ERR_NULL;
    if (ngroups < 1 || ngroups > SAT_ACTOR_POOL_MAX_GROUPS) return SAT_ERR_SIZE;
    for (int k = 0; k < ngroups; ++k)
        if (!groups[k].packed || !groups[k].tc_image || !groups[k].tc_tables) return SAT_ERR_NULL;
    if (wa->in_dim != IN || wa->hidden != HID || wa->act_dim != 3) return SAT_ERR_SIZE;
    if (n <= 0 || ((uintptr_t)wa->packed & 15) || ((uintptr_t)image_a & 15)) return SAT_ERR_SIZE;
    if (!obs_f32 && (st->n < n || st->ld < st->n)) return SAT_ERR_SIZE;
    TcPool pool = {};
    pool.groups = ngroups;
    int64_t lo = 0;
    for (int k = 0; k < ngroups; ++k) {
        const SatActorPoolGroup& g = groups[k];
        const int64_t hi = g.row_end;
        if (hi <= lo || (k + 1 < ngroups && hi % TM) || (k + 1 == ngroups && hi != n)) return SAT_ERR_SIZE;
        if (((uintptr_t)g.packed | (uintptr_t)g.tc_image | (uintptr_t)g.tc_tables) & 15) return SAT_ERR_SIZE;
        if ((g.use_tanh != 0) != (wa->use_tanh != 0)) return SAT_ERR_MODE;      // one activation per launch
        pool.packed[k] = g.packed;
        pool.image[k] = reinterpret_cast<const unsigned char*>(g.tc_image);
        pool.tables[k] = g.tc_tables;
        pool.row_end[k] = hi;
        pool.max_action[k] = g.max_action;
        lo = hi;
    }
    int sms = 0;
    cudaError_t e = (cudaError_t)tc_setup(&sms);
    if (e != cudaSuccess) return (int)e;
    cudaStream_t s = (cudaStream_t)stream;
    TcNet n0 = {wa->packed, reinterpret_cast<unsigned char*>(image_a), nullptr, act_a, logp_a, nullptr, nullptr, step_a, wa->max_action};
    TcNet n1 = {nullptr, nullptr, nullptr, act_b, logp_b, nullptr, nullptr, step_b, 0.0f};
    actor_tc_pack_kernel<<<dim3((NCHUNK * 4 * HID + 255) / 256, 1), 256, 0, s>>>(n0.packed, const_cast<unsigned char*>(n0.image),
                                                                             nullptr, nullptr);
    int rc = launch_status();
    if (rc) return rc;
    SatEnvState s0 = {};
    if (!obs_f32) s0 = *st;
    const int64_t work = ((n + TM - 1) / TM) * 2;
    const unsigned blocks = (unsigned)(work < sms ? work : sms);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = TC_SMEM; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;     // overlap this kernel's prologue with the pack kernel
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    e = wa->use_tanh ? cudaLaunchKernelEx(&cfg, actor_tc_kernel<true, true>, n0, n1, 2, obs_f32, s0, obs_stats, n, row_offset, seed, obs_out, pool)
                     : cudaLaunchKernelEx(&cfg, actor_tc_kernel<false, true>, n0, n1, 2, obs_f32, s0, obs_stats, n, row_offset, seed, obs_out, pool);
    return e == cudaSuccess ? launch_status() : (int)e;
}
}  // namespace

extern "C" {

int sat_actor_sample_tc(const SatActorWeights* w, float* tc_image, const float* obs_f32, const SatEnvState* st,
                        const double* obs_stats, int64_t n, int64_t row_offset, uint64_t seed, uint64_t step,
                        const float* eps_in, float* act, float* logp, float* mean_out, float* eps_out, float* obs_out,
                        void* stream) {
    return launch_tc(w, tc_image, nullptr, nullptr, obs_f32, st, obs_stats, n, row_offset, seed, step, 0, eps_in, act, logp,
                     mean_out, eps_out, obs_out, nullptr, nullptr, stream);
}

int sat_actor_sample_pair_tc(const SatActorWeights* wa, const SatActorWeights* wb, float* tc_image_a, float* tc_image_b,
                             const float* obs_f32, const SatEnvState* st, const double* obs_stats, int64_t n, int64_t row_offset,
                             uint64_t seed, uint64_t step_a, uint64_t step_b, float* act_a, float* logp_a, float* obs_out,
                             float* act_b, float* logp_b, void* stream) {
    if (!wb) return SAT_ERR_NULL;
    return launch_tc(wa, tc_image_a, wb, tc_image_b, obs_f32, st, obs_stats, n, row_offset, seed, step_a, step_b, nullptr, act_a,
                     logp_a, nullptr, nullptr, obs_out, act_b, logp_b, stream);
}

int sat_actor_tc_snapshot(const SatActorWeights* w, float* tc_image, float* tc_tables, SatActorPoolGroup* snap, void* stream) {
    if (!w || !w->packed || !tc_image || !tc_tables || !snap) return SAT_ERR_NULL;
    if (w->in_dim != IN || w->hidden != HID || w->act_dim != 3) return SAT_ERR_SIZE;
    if (((uintptr_t)w->packed | (uintptr_t)tc_image | (uintptr_t)tc_tables) & 15) return SAT_ERR_SIZE;
    cudaStream_t s = (cudaStream_t)stream;
    actor_tc_pack_kernel<<<dim3((NCHUNK * 4 * HID + 255) / 256, 1), 256, 0, s>>>(w->packed, reinterpret_cast<unsigned char*>(tc_image),
                                                                             nullptr, nullptr);
    int rc = launch_status();
    if (rc) return rc;
    actor_tc_table_kernel<<<1, HID, 0, s>>>(w->packed, tc_tables, w->use_tanh);
    rc = launch_status();
    if (rc) return rc;
    *snap = SatActorPoolGroup{w->packed, tc_image, tc_tables, 0, w->use_tanh != 0, w->max_action};
    return SAT_OK;
}

int sat_actor_sample_pool_tc(const SatActorWeights* wa, float* tc_image_a, const SatActorPoolGroup* groups_host, int groups,
                             const float* obs_f32, const SatEnvState* st, const double* obs_stats, int64_t n,
                             int64_t row_offset, uint64_t seed, uint64_t step_a, uint64_t step_b, float* act_a, float* logp_a,
                             float* obs_out, float* act_b, float* logp_b, void* stream) {
    return launch_pool(wa, tc_image_a, groups_host, groups, obs_f32, st, obs_stats, n, row_offset, seed, step_a, step_b, act_a,
                       logp_a, obs_out, act_b, logp_b, stream);
}

}  // extern "C"
