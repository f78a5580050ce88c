// Argument block shared by the AFM kernels (afm.cu: fp32 SIMT; afm_fused_tc.cu: fused tcgen05 training pass).
#pragma once
#include "common.cuh"

namespace hhfm {

constexpr int kAfmMaxF = 16;
constexpr int kAfmMaxP = kAfmMaxF * (kAfmMaxF - 1) / 2;

struct AfmArgs {
  const int32_t* idx;     // [B, F]
  int64_t B;
  int F, K, A, P;
  const float* V;
  const float* bias;
  const float* b0;
  const float* W;         // [K, A]
  const float* batt;      // [A]
  const float* pvec;      // [A]
  const float* wpred;     // [K]
  const float* labels;
  float* out;
  float* gV;
  float* gbias;
  float* gb0;
  float* gW;
  float* gbatt;
  float* gp;
  float* gwpred;
  float* loss_partials;
  int32_t* touch_stamp;
  int32_t stamp;
  int32_t* touched_rows;
  int32_t* touched_count;
  HotPlan hot;
  // training dropout (AFM.py:126,134), read by the DROP instantiations and the attention=0 kernel only:
  // m_p = mask(seed, s, p) / keep_att on the attention weights, n_k = mask(splitmix64(seed), s, k) / keep_vec on the
  // pooled vector, s = sample_base + row (the row's index in the global batch under data parallelism)
  float keep_att, keep_vec;
  uint64_t drop_seed;
  int64_t sample_base;
};

// 0/1 masks of the two AFM dropout streams (oracle: afm_dropout_masks)
__device__ __forceinline__ float afm_mask_att(const AfmArgs& a, int64_t s, int p) {
  return dropout_keep01(a.drop_seed, a.sample_base + s, p, a.keep_att);
}
__device__ __forceinline__ float afm_mask_vec(const AfmArgs& a, uint64_t vseed, int64_t s, int k) {
  return dropout_keep01(vseed, a.sample_base + s, k, a.keep_vec);
}

// afm_fused_tc.cu: returns 1 when the shape is not covered (the caller falls back to the SIMT kernels), else an HHFM_* code.
// drop: the DROP instantiation (keep < 1 on either stream).
int dispatch_afm_fused_tc(const AfmArgs& a, int64_t M, cudaStream_t st, bool drop = false);

}  // namespace hhfm
