// ppo_fb_tc.cuh -- launch interface of the tensor-core forward / backward kernel of the fused PPO step (ppo_fb_tc.cu), used by
// ppo_update.cu. Same inputs, outputs and layouts as ppo_fb_kernel; a row tile is 128 rows (mp must be a multiple of 128) and
// part_head / part_scal hold one entry per 128-row tile. part_stat non-null (actor only) selects the instantiation that also writes
// the per-tile diagnostics part_stat [tile][8] (surrogate, entropy, approximate KL, clipped; ppo_update.cu sums them).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

constexpr int64_t SAT_PPO_TC_IMAGE_BYTES = 34 * 3 * 256 * 32;      // 17 chunks x 2 sub-chunks x [h | m | l] x 256 rows x 32 bytes

int ppo_fb_tc_launch(bool critic, bool use_tanh, const float* packed, unsigned char* image, float max_action, const float* s,
                     const float* a, const float* old_logp, const float* adv, const float* v_target, const int64_t* index,
                     int64_t n, float inv_n, float epsilon, float entropy_coef, float* h1g, float* dz2b, float* dz1g, float* xs,
                     float* part_head, float* part_scal, int64_t mp, float* part_stat, cudaStream_t stream);

// dW2 = dz2^T h1 on the tensor cores (ppo_wgrad2_tc.cu): same operands / output as ppo_wgrad2_kernel; part_w2 [slabs][256][256]
int ppo_wgrad2_tc_launch(const float* dz2b, const float* h1g, int64_t mp, int slabs, float* part_w2, cudaStream_t stream);
