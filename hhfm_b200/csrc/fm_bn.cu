// FM with batch normalisation of the interaction vector (FM.py:111-112, batch_norm=1):
//   x = 0.5 (S^2 - sum_f e_f^2)  [B, K],  y = gamma (x - mu) / sqrt(var + eps) + beta,  z = y / keep * m,
//   out = sum_k z + sum_f b[x_f] + b0,
// the batch statistics (mu, var) taken over the whole batch (tf.contrib.layers.batch_norm, is_training=True).  The
// statistics sit between the forward and the backward of every sample, so the training step is five launches:
//   1. fm_bn_gather_kernel   rows -> x and sum_f b[x_f] into the workspace; per-CTA (n, mean, M2) per column (Welford
//                            per lane, Chan's formula across the CTA's lane groups in a fixed order)
//   2. fm_bn_reduce_kernel<true>   the CTA partials in a fixed order (Chan, in double) -> mu, 1/sqrt(var + eps); the
//                            moving statistics move towards mu and the Bessel-corrected variance
//   3. fm_bn_loss_kernel     x -> out, the loss partials and g = out - y per sample; per-CTA sums of d and d * xhat per
//                            column (d = g m / keep) and of g
//   4. fm_bn_reduce_kernel<false>  those partials in a fixed order -> d beta, d gamma, d b0
//   5. fm_bn_scatter_kernel  rows gathered again, x recomputed, dx = gamma / sqrt(var + eps) (d - dbeta/B - xhat dgamma/B),
//                            gV[x_f] += dx (S - e_f), gbias[x_f] += g with the hot-row plan and the touched-row list
// Every value that leaves the step except the row gradients (float atomics, as in fm_kernel) is a fixed-order reduction,
// so the batch statistics, the loss, d gamma, d beta, d b0 and the moving statistics are bit-identical from run to run.
// Synchronised batch norm (data parallelism, DESIGN.md 7) runs the same passes as three phases with an all-gather of one
// small double vector per rank between them: passes 2 and 4 stop before finalising and write this rank's merged
// (n, mean, M2) / (sum g, sum d, sum d xhat); the next phase merges the gathered vectors of all ranks in rank order
// (fm_bn_rank_merge_kernel) and finalises with the same code as the single call.  With one rank the phases reproduce
// the single call bit for bit: a double partial merged into an empty state is itself.
// Lane mapping: fm.cu's Frag<LPS, VPL> (one sample per aligned group of LPS lanes, VPL float4 per lane).
#include <math.h>

#include "common.cuh"

namespace hhfm {

struct FmBnArgs {
  const int32_t* col;
  int64_t B;
  int F, K;
  const float* V;
  const float* bias;
  const float* b0;
  const float* labels;
  float* out;
  float* gV;
  float* gbias;
  float* gb0;
  float* loss_partials;
  int32_t* touch_stamp;
  int32_t stamp;
  int32_t* touched_rows;
  int32_t* touched_count;
  HotPlan hot;
  int groups_active;
  float keep;
  uint64_t drop_seed;
  const float* gamma;
  const float* beta;
  float* mm;         // moving mean [K]
  float* mv;         // moving variance [K]
  float* dgamma;
  float* dbeta;
  float eps, decay;
  // workspace
  float* x;          // [B, K]
  float* bsum;       // [B]  sum_f b[x_f]
  float* g;          // [B]  d loss / d out
  float* part;       // [kPartials, 2K + 1]: pass 1 (mean, M2, n), pass 3 (sum d, sum d xhat, sum g) per CTA
  float* colv;       // [5, K]: mu, 1/sqrt(var + eps), gamma/sqrt(var + eps), dbeta / B, dgamma / B
  int64_t* glob;     // synchronised phases only (NULL in the single call): [global batch size, global index of sample 0]
};

static inline size_t bn_align(size_t b) { return (b + 255) / 256 * 256; }

static size_t fm_bn_ws_bytes(int64_t B, int64_t K) {
  return bn_align((size_t)B * K * 4) + 2 * bn_align((size_t)B * 4) + bn_align((size_t)kPartials * (2 * K + 1) * 4) +
         bn_align((size_t)5 * K * 4);
}

// the synchronised phases: the same layout plus the global batch size and index base
static size_t fm_bn_sync_ws_bytes(int64_t B, int64_t K) { return fm_bn_ws_bytes(B, K) + bn_align(2 * sizeof(int64_t)); }

static void fm_bn_ws_bind(FmBnArgs& a, void* ws, bool sync = false) {
  char* p = static_cast<char*>(ws);
  a.x = reinterpret_cast<float*>(p);     p += bn_align((size_t)a.B * a.K * 4);
  a.bsum = reinterpret_cast<float*>(p);  p += bn_align((size_t)a.B * 4);
  a.g = reinterpret_cast<float*>(p);     p += bn_align((size_t)a.B * 4);
  a.part = reinterpret_cast<float*>(p);  p += bn_align((size_t)kPartials * (2 * a.K + 1) * 4);
  a.colv = reinterpret_cast<float*>(p);  p += bn_align((size_t)5 * a.K * 4);
  a.glob = sync ? reinterpret_cast<int64_t*>(p) : nullptr;
}

__device__ __forceinline__ float4 f4_div(float4 a, float s) { return make_float4(a.x / s, a.y / s, a.z / s, a.w / s); }

// S = sum_f e_f, Q = sum_f e_f^2 over the fields in order (4 gathers in flight), and the bias sum, as fm_kernel.
template <int LPS, int VPL>
__device__ __forceinline__ void bn_gather(const FmBnArgs& a, int64_t s, bool valid, int lg, Frag<LPS, VPL>& S, Frag<LPS, VPL>& Q,
                                          float& bsum) {
  frag_zero(S);
  frag_zero(Q);
  bsum = 0.f;
  const int64_t beg = valid ? s * a.F : 0, end = valid ? beg + a.F : 0;
  for (int64_t j = beg; j < end; j += 4) {
    int id[4];
    Frag<LPS, VPL> e[4];
#pragma unroll
    for (int u = 0; u < 4; u++) id[u] = (j + u) < end ? __ldg(a.col + j + u) : -1;
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (id[u] >= 0) frag_load(e[u], a.V, id[u], a.K, lg);
#pragma unroll
    for (int u = 0; u < 4; u++) {
      if (id[u] >= 0) {
        if (a.bias) bsum += __ldg(a.bias + id[u]);
#pragma unroll
        for (int i = 0; i < VPL; i++) {
          S.v[i] = f4_add(S.v[i], e[u].v[i]);
          Q.v[i] = f4_add(Q.v[i], f4_mul(e[u].v[i], e[u].v[i]));
        }
      }
    }
  }
}

__device__ __forceinline__ float4 bn_interaction(float4 S, float4 Q) { return f4_scale(f4_sub(f4_mul(S, S), Q), 0.5f); }

__device__ __forceinline__ float4 bn_mask(const FmBnArgs& a, int64_t s, int k0) {
  return make_float4(dropout_keep01(a.drop_seed, s, k0, a.keep), dropout_keep01(a.drop_seed, s, k0 + 1, a.keep),
                     dropout_keep01(a.drop_seed, s, k0 + 2, a.keep), dropout_keep01(a.drop_seed, s, k0 + 3, a.keep));
}

__device__ __forceinline__ void chan_merge(float& n, float& mean, float& m2, float nb, float mb, float m2b) {
  if (nb == 0.f) return;
  const float nn = n + nb, d = mb - mean;
  mean = mean + d * (nb / nn);
  m2 = m2 + m2b + d * d * (n * nb / nn);
  n = nn;
}

// Chan's formula in double: the merge of CTA partials (pass 2) and of the ranks' partials (synchronised phases)
__device__ __forceinline__ void chan_merge_d(double& n, double& mean, double& m2, double nb, double mb, double m2b) {
  if (nb == 0.0) return;
  const double nn = n + nb, d = mb - mean;
  mean += d * (nb / nn);
  m2 += m2b + d * d * (n * nb / nn);
  n = nn;
}

// Global index of local sample 0 for the dropout mask: the synchronised phases draw the mask of the sample's index in the
// global batch (the sizes of the lower ranks before it); the single call starts at 0.
__device__ __forceinline__ int64_t bn_index_base(const FmBnArgs& a) { return a.glob ? a.glob[1] : 0; }

// Column c from the merged (n, mean, M2) of the batch: mu, 1/sqrt(var + eps), gamma/sqrt(var + eps); the moving statistics
// move towards mu and the Bessel-corrected variance.  Biased batch variance for the normalisation, n - 1 taken as 1 when
// n = 1 (the fused batch-norm kernel of tf.contrib.layers.batch_norm, DESIGN.md 7).  An empty batch leaves the layer as is.
__device__ __forceinline__ void bn_finish_stats(const FmBnArgs& a, int c, double n, double mean, double m2) {
  const int K = a.K;
  if (n == 0.0) {
    a.colv[c] = 0.f;
    a.colv[K + c] = 0.f;
    a.colv[2 * K + c] = 0.f;
    return;
  }
  const float mu = (float)mean, var = (float)(m2 / n);
  const float var_u = (float)(m2 / (n > 1.0 ? n - 1.0 : 1.0));
  const float is = 1.f / sqrtf(var + a.eps);
  const float f = 1.f - a.decay;
  a.mm[c] = a.mm[c] - (a.mm[c] - mu) * f;
  a.mv[c] = a.mv[c] - (a.mv[c] - var_u) * f;
  a.colv[c] = mu;
  a.colv[K + c] = is;
  a.colv[2 * K + c] = a.gamma[c] * is;
}

// Column c from the batch sums of d and d xhat: d beta, d gamma and their means over the n samples of the batch.
__device__ __forceinline__ void bn_finish_sums(const FmBnArgs& a, int c, double n, double sd, double sdx) {
  const int K = a.K;
  const float db = (float)sd, dg = (float)sdx;
  a.dbeta[c] = db;
  a.dgamma[c] = dg;
  a.colv[3 * K + c] = n > 0.0 ? db / (float)n : 0.f;
  a.colv[4 * K + c] = n > 0.0 ? dg / (float)n : 0.f;
}

// ---- pass 1 -----------------------------------------------------------------------------------------------------
template <int LPS, int VPL>
__global__ void __launch_bounds__(kBlock) fm_bn_gather_kernel(const FmBnArgs a) {
  constexpr int G = 32 / LPS, NG = (kBlock / 32) * G, KC = 4 * LPS * VPL;
  __shared__ float4 sh_a[NG * KC / 4], sh_b[NG * KC / 4];
  __shared__ float sh_n[NG];
  using F4 = Frag<LPS, VPL>;
  const int lane = threadIdx.x & 31, lg = lane % LPS, grp = lane / LPS, gi = (threadIdx.x >> 5) * G + grp;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int K = a.K, kv = K >> 2;
  F4 mean, m2;
  frag_zero(mean);
  frag_zero(m2);
  int n = 0;
  for (int64_t s0 = warp_g * G; s0 < a.B; s0 += n_warps * G) {
    const int64_t s = s0 + grp;
    const bool valid = s < a.B;
    F4 S, Q;
    float bsum;
    bn_gather(a, s, valid, lg, S, Q, bsum);
    if (!valid) continue;
    n++;
    const float inv = 1.f / (float)n;
#pragma unroll
    for (int i = 0; i < VPL; i++) {
      const int c = lg + i * LPS;
      if (c < kv) {
        const float4 x = bn_interaction(S.v[i], Q.v[i]);
        reinterpret_cast<float4*>(a.x + s * K)[c] = x;
        const float4 d = f4_sub(x, mean.v[i]);
        mean.v[i] = f4_add(mean.v[i], f4_scale(d, inv));
        m2.v[i] = f4_add(m2.v[i], f4_mul(d, f4_sub(x, mean.v[i])));
      }
    }
    if (lg == 0) a.bsum[s] = bsum;
  }
#pragma unroll
  for (int i = 0; i < VPL; i++) {
    sh_a[gi * (KC / 4) + lg + i * LPS] = mean.v[i];
    sh_b[gi * (KC / 4) + lg + i * LPS] = m2.v[i];
  }
  if (lg == 0) sh_n[gi] = (float)n;
  __syncthreads();
  const float* fa = reinterpret_cast<const float*>(sh_a);
  const float* fb = reinterpret_cast<const float*>(sh_b);
  float* p = a.part + (size_t)blockIdx.x * (2 * K + 1);
  float nt = 0.f;
  for (int c = threadIdx.x; c < K; c += blockDim.x) {
    float nn = 0.f, mu = 0.f, M2 = 0.f;
    for (int q = 0; q < NG; q++) chan_merge(nn, mu, M2, sh_n[q], fa[q * KC + c], fb[q * KC + c]);
    p[c] = mu;
    p[K + c] = M2;
    nt = nn;
  }
  if (threadIdx.x == 0) p[2 * K] = nt;
}

// ---- pass 3 -----------------------------------------------------------------------------------------------------
template <int LPS, int VPL, bool DROP>
__global__ void __launch_bounds__(kBlock, 1) fm_bn_loss_kernel(const FmBnArgs a) {
  constexpr int G = 32 / LPS, NG = (kBlock / 32) * G, KC = 4 * LPS * VPL;
  __shared__ float4 sh_a[NG * KC / 4], sh_b[NG * KC / 4];
  __shared__ float sh_n[NG];
  __shared__ float scratch[32];
  using F4 = Frag<LPS, VPL>;
  const int lane = threadIdx.x & 31, lg = lane % LPS, grp = lane / LPS, gi = (threadIdx.x >> 5) * G + grp;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int K = a.K, kv = K >> 2;
  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  F4 mu, is, ga, be, acc_b, acc_g;
  frag_zero(acc_b);
  frag_zero(acc_g);
  frag_load(mu, a.colv, 0, K, lg);
  frag_load(is, a.colv, 1, K, lg);
  frag_load(ga, a.gamma, 0, K, lg);
  frag_load(be, a.beta, 0, K, lg);
  float loss_acc = 0.f, g_acc = 0.f;
  const int64_t sb = bn_index_base(a);
  for (int64_t s0 = warp_g * G; s0 < a.B; s0 += n_warps * G) {
    const int64_t s = s0 + grp;
    const bool valid = s < a.B;
    F4 x, xh, m;
    frag_load(x, a.x, valid ? s : 0, K, lg);
    float part = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; i++) {
      xh.v[i] = f4_mul(f4_sub(x.v[i], mu.v[i]), is.v[i]);
      float4 z = f4_add(f4_mul(ga.v[i], xh.v[i]), be.v[i]);         // zero in the padding columns (gamma, beta read 0)
      if constexpr (DROP) {
        m.v[i] = bn_mask(a, sb + (valid ? s : 0), 4 * (lg + i * LPS));
        z = f4_mul(f4_div(z, a.keep), m.v[i]);
      }
      part += f4_hsum(z);
    }
    const float bil = group_sum<LPS>(part);
    if (!valid) continue;
    const float out = (bil + __ldg(a.bsum + s)) + b0;
    const float diff = __ldg(a.labels + s) - out;
    const float g = -diff;
    if (lg == 0) {
      loss_acc += 0.5f * diff * diff;
      g_acc += g;
      a.g[s] = g;
      if (a.out) a.out[s] = out;
    }
#pragma unroll
    for (int i = 0; i < VPL; i++) {
      float4 d = make_float4(g, g, g, g);
      if constexpr (DROP) d = f4_mul(d, f4_div(m.v[i], a.keep));
      if (lg + i * LPS < kv) {
        acc_b.v[i] = f4_add(acc_b.v[i], d);
        acc_g.v[i] = f4_add(acc_g.v[i], f4_mul(d, xh.v[i]));
      }
    }
  }
#pragma unroll
  for (int i = 0; i < VPL; i++) {
    sh_a[gi * (KC / 4) + lg + i * LPS] = acc_b.v[i];
    sh_b[gi * (KC / 4) + lg + i * LPS] = acc_g.v[i];
  }
  if (lg == 0) sh_n[gi] = g_acc;
  __syncthreads();
  const float* fa = reinterpret_cast<const float*>(sh_a);
  const float* fb = reinterpret_cast<const float*>(sh_b);
  float* p = a.part + (size_t)blockIdx.x * (2 * K + 1);
  for (int c = threadIdx.x; c < K; c += blockDim.x) {
    float sb = 0.f, sg = 0.f;
    for (int q = 0; q < NG; q++) {
      sb += fa[q * KC + c];
      sg += fb[q * KC + c];
    }
    p[c] = sb;
    p[K + c] = sg;
  }
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int q = 0; q < NG; q++) t += sh_n[q];
    p[2 * K] = t;
  }
  const float bl = block_sum(loss_acc, scratch);
  write_partial(a.loss_partials, bl);
}

// ---- passes 2 and 4: the CTA partials of `n_part` CTAs, one CTA, fixed order --------------------------------------
// Thread t takes column c = cb + t % cols and the partials seg, seg + nseg, ... (seg = t / cols); the nseg segment results
// of a column are merged in segment order by the thread of segment 0.  vec == NULL: finalised for this batch (the single
// call).  Otherwise the merged partials go to vec [2K + 1] as doubles for the all-gather of the synchronised phases:
// pass 2 (n, mean[K], M2[K]), pass 4 (sum g, sum d[K], sum d xhat[K]).
constexpr int kReduceThreads = 1024;     // one CTA does the whole merge: more threads, fewer partials each

template <bool STATS>
__global__ void __launch_bounds__(kReduceThreads) fm_bn_reduce_kernel(const FmBnArgs a, int n_part, double* vec) {
  __shared__ double sh[3][kReduceThreads];
  const int K = a.K, W = 2 * K + 1;
  const int cols = K < (int)blockDim.x ? K : (int)blockDim.x;
  const int nseg = blockDim.x / cols;
  const int seg = threadIdx.x / cols;
  for (int cb = 0; cb < K; cb += cols) {
    const int c = cb + threadIdx.x % cols;
    double r0 = 0.0, r1 = 0.0, r2 = 0.0;       // STATS: n, mean, M2;  else: sum d, sum d xhat
    if (seg < nseg && c < K) {
      for (int p = seg; p < n_part; p += nseg) {
        const float* q = a.part + (size_t)p * W;
        if (STATS) {
          chan_merge_d(r0, r1, r2, q[2 * K], q[c], q[K + c]);
        } else {
          r0 += q[c];
          r1 += q[K + c];
        }
      }
    }
    if (seg < nseg) {
      sh[0][threadIdx.x] = r0;
      sh[1][threadIdx.x] = r1;
      sh[2][threadIdx.x] = r2;
    }
    __syncthreads();
    if (seg == 0 && c < K) {
      for (int t = 1; t < nseg; t++) {
        const int o = t * cols + threadIdx.x;
        if (STATS) {
          chan_merge_d(r0, r1, r2, sh[0][o], sh[1][o], sh[2][o]);
        } else {
          r0 += sh[0][o];
          r1 += sh[1][o];
        }
      }
      if (vec != nullptr) {
        if (STATS && c == 0) vec[0] = r0;
        vec[1 + c] = STATS ? r1 : r0;
        vec[1 + K + c] = STATS ? r2 : r1;
      } else if (STATS) {
        bn_finish_stats(a, c, (double)a.B, r1, r2);
      } else {
        bn_finish_sums(a, c, (double)a.B, r0, r1);
      }
    }
    __syncthreads();
  }
  if (!STATS && threadIdx.x == 0 && (a.gb0 != nullptr || vec != nullptr)) {
    double t = 0.0;
    for (int p = 0; p < n_part; p++) t += a.part[(size_t)p * W + 2 * K];
    if (a.gb0 != nullptr) *a.gb0 += (float)t;
    if (vec != nullptr) vec[0] = t;
  }
}

// ---- synchronised phases: the gathered per-rank vectors [n_ranks, 2K + 1], merged in rank order, one CTA ------------
// STATS: (n, mean, M2) of every rank (Chan) -> finalised as pass 2 does for the global batch; thread 0 records the global
// batch size and the global index of this rank's first sample.  Else: the sums of d and d xhat of every rank -> d beta,
// d gamma and their means over the global batch.
template <bool STATS>
__global__ void __launch_bounds__(kReduceThreads) fm_bn_rank_merge_kernel(const FmBnArgs a, const double* all, int n_ranks,
                                                                          int rank) {
  const int K = a.K, W = 2 * K + 1;
  if (STATS && threadIdx.x == 0) {
    int64_t n = 0, base = 0;
    for (int r = 0; r < n_ranks; r++) {
      const int64_t nr = (int64_t)all[(size_t)r * W];
      if (r < rank) base += nr;
      n += nr;
    }
    a.glob[0] = n;
    a.glob[1] = base;
  }
  const double n_glob = STATS ? 0.0 : (double)a.glob[0];      // written by the STATS merge of this step
  for (int c = threadIdx.x; c < K; c += blockDim.x) {
    double r0 = 0.0, r1 = 0.0, r2 = 0.0;
    for (int r = 0; r < n_ranks; r++) {
      const double* v = all + (size_t)r * W;
      if (STATS) {
        chan_merge_d(r0, r1, r2, v[0], v[1 + c], v[1 + K + c]);
      } else {
        r0 += v[1 + c];
        r1 += v[1 + K + c];
      }
    }
    if (STATS)
      bn_finish_stats(a, c, r0, r1, r2);
    else
      bn_finish_sums(a, c, n_glob, r0, r1);
  }
}

// ---- pass 5 -----------------------------------------------------------------------------------------------------
template <int LPS, int VPL, bool DROP>
__global__ void __launch_bounds__(kBlock) fm_bn_scatter_kernel(const FmBnArgs a) {
  using F4 = Frag<LPS, VPL>;
  const int lane = threadIdx.x & 31, lg = lane % LPS, grp = lane / LPS;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int ga = a.groups_active;
  const int K = a.K, kv = K >> 2;
  const int rep = a.hot.slot ? (int)((warp_g * (32 / LPS) + grp) % a.hot.n_rep) : 0;
  const float4* cv = reinterpret_cast<const float4*>(a.colv);
  const int64_t sb = bn_index_base(a);
  for (int64_t s0 = warp_g * ga; s0 < a.B; s0 += n_warps * ga) {
    const int64_t s = s0 + grp;
    const bool valid = (grp < ga) && (s < a.B);
    if (!valid) continue;
    F4 S, Q, dx;
    float bsum;
    bn_gather(a, s, true, lg, S, Q, bsum);
    const float g = __ldg(a.g + s);
#pragma unroll
    for (int i = 0; i < VPL; i++) {
      const int c = lg + i * LPS;
      dx.v[i] = f4_zero();
      if (c < kv) {
        const float4 xh = f4_mul(f4_sub(bn_interaction(S.v[i], Q.v[i]), ldg4(cv + c)), ldg4(cv + kv + c));
        const float4 d = DROP ? f4_mul(make_float4(g, g, g, g), f4_div(bn_mask(a, sb + s, 4 * c), a.keep)) : make_float4(g, g, g, g);
        dx.v[i] = f4_mul(ldg4(cv + 2 * kv + c), f4_sub(f4_sub(d, ldg4(cv + 3 * kv + c)), f4_mul(xh, ldg4(cv + 4 * kv + c))));
      }
    }
    // ---- gV[x_f] += dx * (S - e_f); gbias[x_f] += g ----
    const int64_t beg = s * a.F, end = beg + a.F;
    for (int64_t j = beg; j < end; j += 4) {
      int id[4];
      F4 e[4];
#pragma unroll
      for (int u = 0; u < 4; u++) id[u] = (j + u) < end ? __ldg(a.col + j + u) : -1;
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (id[u] >= 0) frag_load(e[u], a.V, id[u], K, lg);
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if (id[u] >= 0) {
          F4 d;
#pragma unroll
          for (int i = 0; i < VPL; i++) d.v[i] = f4_mul(dx.v[i], f4_sub(S.v[i], e[u].v[i]));
          scatter_row<LPS, VPL>(a.gV, a.hot, rep, id[u], K, lg, d);
          if (lg == 0) {
            if (a.gbias) scatter_bias(a.gbias, a.hot, rep, id[u], g);
            touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, id[u]);
          }
        }
      }
    }
  }
}

// ---- inference (train_phase=False): the moving statistics, no dropout --------------------------------------------
template <int LPS, int VPL>
__global__ void __launch_bounds__(kBlock) fm_bn_fwd_kernel(const FmBnArgs a) {
  using F4 = Frag<LPS, VPL>;
  const int lane = threadIdx.x & 31, lg = lane % LPS, grp = lane / LPS;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  constexpr int G = 32 / LPS;
  const int K = a.K;
  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  F4 sc, mm, be;                                    // sc = gamma / sqrt(mv + eps); zero in the padding columns
  frag_load(sc, a.gamma, 0, K, lg);
  frag_load(mm, a.mm, 0, K, lg);
  frag_load(be, a.beta, 0, K, lg);
  {
    F4 mv;
    frag_load(mv, a.mv, 0, K, lg);
#pragma unroll
    for (int i = 0; i < VPL; i++)
      sc.v[i] = make_float4(sc.v[i].x / sqrtf(mv.v[i].x + a.eps), sc.v[i].y / sqrtf(mv.v[i].y + a.eps),
                            sc.v[i].z / sqrtf(mv.v[i].z + a.eps), sc.v[i].w / sqrtf(mv.v[i].w + a.eps));
  }
  for (int64_t s0 = warp_g * G; s0 < a.B; s0 += n_warps * G) {
    const int64_t s = s0 + grp;
    const bool valid = s < a.B;
    F4 S, Q;
    float bsum;
    bn_gather(a, s, valid, lg, S, Q, bsum);
    float part = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; i++)
      part += f4_hsum(f4_add(f4_mul(sc.v[i], f4_sub(bn_interaction(S.v[i], Q.v[i]), mm.v[i])), be.v[i]));
    const float bil = group_sum<LPS>(part);
    if (valid && lg == 0) a.out[s] = (bil + bsum) + b0;
  }
}

template <class KERN>
static int bn_grid(KERN k, int64_t B, int lps) {
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, kBlock, 0);
  if (occ < 1) occ = 1;
  return grid_for(B, (kBlock / 32) * (32 / lps), occ);
}

// CTAs per SM of passes 1, 3 and 5 (the grid is this times the SMs, capped by B)
struct BnCaps {
  int g1, g3, g5;
};

template <int LPS, int VPL, bool DROP>
static const BnCaps& bn_caps() {
  static const BnCaps c{bn_grid(fm_bn_gather_kernel<LPS, VPL>, (int64_t)1 << 40, LPS),
                        bn_grid(fm_bn_loss_kernel<LPS, VPL, DROP>, (int64_t)1 << 40, LPS),
                        bn_grid(fm_bn_scatter_kernel<LPS, VPL, DROP>, (int64_t)1 << 40, LPS)};
  return c;
}

// CTAs of a pass over B samples: one per (kBlock / 32) * (32 / LPS) samples, at most `cap`, at least one (an empty rank
// of the synchronised phases still writes its zero partials)
static int bn_ctas(int64_t B, int lps, int cap) {
  const int64_t per_cta = (kBlock / 32) * (32 / lps);
  const int64_t need = (B + per_cta - 1) / per_cta;
  return need < 1 ? 1 : (int)(need < cap ? need : cap);
}

template <int LPS, int VPL, bool DROP>
static void launch_fm_bn_scatter(FmBnArgs a, int deterministic, cudaStream_t st) {
  if (deterministic) {                          // one warp in program order: bit-reproducible row gradients
    a.groups_active = 1;
    fm_bn_scatter_kernel<LPS, VPL, DROP><<<1, 32, 0, st>>>(a);
  } else {
    a.groups_active = 32 / LPS;
    fm_bn_scatter_kernel<LPS, VPL, DROP><<<bn_ctas(a.B, LPS, bn_caps<LPS, VPL, DROP>().g5), kBlock, 0, st>>>(a);
  }
}

template <int LPS, int VPL, bool DROP>
static int launch_fm_bn_train(FmBnArgs a, int deterministic, cudaStream_t st) {
  const BnCaps& cap = bn_caps<LPS, VPL, DROP>();
  const int n1 = bn_ctas(a.B, LPS, cap.g1), n3 = bn_ctas(a.B, LPS, cap.g3);
  fm_bn_gather_kernel<LPS, VPL><<<n1, kBlock, 0, st>>>(a);
  fm_bn_reduce_kernel<true><<<1, kReduceThreads, 0, st>>>(a, n1, nullptr);
  fm_bn_loss_kernel<LPS, VPL, DROP><<<n3, kBlock, 0, st>>>(a);
  fm_bn_reduce_kernel<false><<<1, kReduceThreads, 0, st>>>(a, n3, nullptr);
  launch_fm_bn_scatter<LPS, VPL, DROP>(a, deterministic, st);
  return check_launch("fm_bn training kernels");
}

// synchronised phase 1: pass 1 and the merge of pass 2 into this rank's (n, mean, M2)
template <int LPS, int VPL>
static int launch_fm_bn_sync_stats(const FmBnArgs& a, double* stats, cudaStream_t st) {
  const int n1 = bn_ctas(a.B, LPS, bn_caps<LPS, VPL, false>().g1);
  fm_bn_gather_kernel<LPS, VPL><<<n1, kBlock, 0, st>>>(a);
  fm_bn_reduce_kernel<true><<<1, kReduceThreads, 0, st>>>(a, n1, stats);
  return check_launch("fm_bn_sync_stats kernels");
}

// synchronised phase 2: the ranks' statistics merged and finalised, pass 3, the merge of pass 4 into this rank's sums
template <int LPS, int VPL, bool DROP>
static int launch_fm_bn_sync_loss(const FmBnArgs& a, const double* stats_all, int n_ranks, int rank, double* sums,
                                  cudaStream_t st) {
  const int n3 = bn_ctas(a.B, LPS, bn_caps<LPS, VPL, DROP>().g3);
  fm_bn_rank_merge_kernel<true><<<1, kReduceThreads, 0, st>>>(a, stats_all, n_ranks, rank);
  fm_bn_loss_kernel<LPS, VPL, DROP><<<n3, kBlock, 0, st>>>(a);
  fm_bn_reduce_kernel<false><<<1, kReduceThreads, 0, st>>>(a, n3, sums);
  return check_launch("fm_bn_sync_loss kernels");
}

// synchronised phase 3: the ranks' sums added in rank order, pass 5
template <int LPS, int VPL, bool DROP>
static int launch_fm_bn_sync_scatter(const FmBnArgs& a, const double* sums_all, int n_ranks, int deterministic,
                                     cudaStream_t st) {
  fm_bn_rank_merge_kernel<false><<<1, kReduceThreads, 0, st>>>(a, sums_all, n_ranks, 0);
  launch_fm_bn_scatter<LPS, VPL, DROP>(a, deterministic, st);
  return check_launch("fm_bn_sync_scatter kernels");
}

template <int LPS, int VPL>
static int launch_fm_bn_fwd(const FmBnArgs& a, cudaStream_t st) {
  static int grid_cap = 0;
  if (grid_cap == 0) grid_cap = bn_grid(fm_bn_fwd_kernel<LPS, VPL>, (int64_t)1 << 40, LPS);
  const int64_t per_cta = (kBlock / 32) * (32 / LPS);
  const int64_t need = (a.B + per_cta - 1) / per_cta;
  fm_bn_fwd_kernel<LPS, VPL><<<(int)(need < grid_cap ? need : grid_cap), kBlock, 0, st>>>(a);
  return check_launch("fm_bn_fwd_kernel");
}

static int check_bn_rows(int64_t B, int64_t F, const void* col, const void* V, int64_t M, int64_t K) {
  HHFM_REQUIRE(B >= 0 && M > 0, "fm_bn: bad sizes B=%lld M=%lld", (long long)B, (long long)M);
  HHFM_REQUIRE(col != nullptr && V != nullptr, "fm_bn: col and V must not be NULL");
  HHFM_REQUIRE(K > 0 && K % 4 == 0 && K <= 512, "fm_bn: K=%lld unsupported (need K %% 4 == 0, K <= 512)", (long long)K);
  HHFM_REQUIRE(F > 0, "fm_bn: F=%lld, need F > 0", (long long)F);
  HHFM_REQUIRE(((uintptr_t)V & 15) == 0, "fm_bn: V must be 16-byte aligned");
  return HHFM_OK;
}

static int check_bn_layer(const float* gamma, const float* beta, const float* mm, const float* mv, float eps) {
  HHFM_REQUIRE(gamma && beta && mm && mv, "fm_bn: gamma, beta, moving_mean and moving_var must not be NULL");
  HHFM_REQUIRE((((uintptr_t)gamma | (uintptr_t)beta | (uintptr_t)mm | (uintptr_t)mv) & 15) == 0,
               "fm_bn: gamma, beta, moving_mean and moving_var must be 16-byte aligned");
  HHFM_REQUIRE(eps > 0.f && eps < INFINITY, "fm_bn: eps must be > 0 (got %g)", (double)eps);
  return HHFM_OK;
}

static int check_bn_common(int64_t B, int64_t F, const void* col, const void* V, int64_t M, int64_t K, const float* gamma,
                           const float* beta, const float* mm, const float* mv, float eps) {
  int rc = check_bn_rows(B, F, col, V, M, K);
  return rc ? rc : check_bn_layer(gamma, beta, mm, mv, eps);
}

static int check_bn_scatter(const int32_t* touch_stamp, int32_t* touched_rows, int32_t* touched_count, const int32_t* hot_slot,
                            float* ghot, int32_t n_rep, int32_t n_hot, const float* gV, float keep) {
  HHFM_REQUIRE(!hot_slot || (ghot && n_rep >= 1 && n_hot >= 1), "fm_bn: hot_slot needs ghot, n_rep, n_hot");
  HHFM_REQUIRE(!touch_stamp || (touched_rows && touched_count), "fm_bn: touch_stamp needs touched_rows/count");
  HHFM_REQUIRE(((uintptr_t)gV & 15) == 0, "fm_bn: gV must be 16-byte aligned");
  HHFM_REQUIRE(keep > 0.f && keep <= 1.f, "fm_bn: dropout keep must be in (0, 1]");
  return HHFM_OK;
}

// the arguments every synchronised phase shares: the batch (B may be 0: an empty rank takes part in both all-gathers),
// the rank layout and the workspace
static int check_bn_sync(const char* what, int64_t B, int64_t K, int32_t n_ranks, int32_t rank, const void* vec,
                         const void* workspace, int64_t workspace_bytes) {
  HHFM_REQUIRE(B >= 0, "%s: bad size B=%lld", what, (long long)B);
  HHFM_REQUIRE(K > 0 && K % 4 == 0 && K <= 512, "%s: K=%lld unsupported (need K %% 4 == 0, K <= 512)", what, (long long)K);
  HHFM_REQUIRE(n_ranks >= 1, "%s: n_ranks=%d, need n_ranks >= 1", what, (int)n_ranks);
  HHFM_REQUIRE(rank >= 0 && rank < n_ranks, "%s: rank=%d outside [0, n_ranks=%d)", what, (int)rank, (int)n_ranks);
  HHFM_REQUIRE(vec != nullptr, "%s: the per-rank vector must not be NULL", what);
  HHFM_REQUIRE(((uintptr_t)vec & 7) == 0, "%s: the per-rank vector must be 8-byte aligned", what);
  const int64_t need = (int64_t)fm_bn_sync_ws_bytes(B, K);
  HHFM_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 15) == 0, "%s: workspace must be non-NULL and 16-byte aligned", what);
  HHFM_REQUIRE(workspace_bytes >= need, "%s: workspace of %lld bytes, need %lld (hhfm_workspace_bytes_fm_bn_sync)", what,
               (long long)workspace_bytes, (long long)need);
  return HHFM_OK;
}

}  // namespace hhfm

using namespace hhfm;

extern "C" int64_t hhfm_workspace_bytes_fm_bn(int64_t B, int64_t K) {
  if (B < 0 || K <= 0 || K > 512) return -1;
  return (int64_t)fm_bn_ws_bytes(B, K);
}

extern "C" int hhfm_fm_bn_fwd_bwd_sqloss(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B, int64_t F,
                                         const float* V, const float* bias, const float* b0, int64_t M, int64_t K,
                                         int32_t interaction, const float* labels, float* out, float* gV, float* gbias,
                                         float* gb0, float* loss_partials, int32_t* touch_stamp, int32_t stamp,
                                         int32_t* touched_rows, int32_t* touched_count, const int32_t* hot_slot, float* ghot,
                                         float* ghot_bias, int32_t n_rep, int32_t n_hot, int32_t deterministic, float keep,
                                         uint64_t drop_seed, const float* gamma, const float* beta, float* moving_mean,
                                         float* moving_var, float* dgamma, float* dbeta, float eps, float decay,
                                         void* workspace, int64_t workspace_bytes, hhfm_stream_t stream) {
  int rc = check_bn_common(B, F, col, V, M, K, gamma, beta, moving_mean, moving_var, eps);
  if (rc) return rc;
  HHFM_REQUIRE(row_ptr == nullptr && val == nullptr, "fm_bn: fixed-width rows only (row_ptr and val must be NULL)");
  HHFM_REQUIRE(interaction == 0, "fm_bn: batch normalisation is on the FM interaction vector (interaction must be 0)");
  HHFM_REQUIRE(labels && gV && loss_partials, "fm_bn: labels, gV and loss_partials are required");
  HHFM_REQUIRE(dgamma && dbeta, "fm_bn: dgamma and dbeta must not be NULL");
  HHFM_REQUIRE(B > 0, "fm_bn: empty batch");
  rc = check_bn_scatter(touch_stamp, touched_rows, touched_count, hot_slot, ghot, n_rep, n_hot, gV, keep);
  if (rc) return rc;
  HHFM_REQUIRE(decay >= 0.f && decay < 1.f, "fm_bn: decay must be in [0, 1) (got %g)", (double)decay);
  const int64_t need = (int64_t)fm_bn_ws_bytes(B, K);
  HHFM_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 15) == 0, "fm_bn: workspace must be non-NULL and 16-byte aligned");
  HHFM_REQUIRE(workspace_bytes >= need, "fm_bn: workspace of %lld bytes, need %lld (hhfm_workspace_bytes_fm_bn)",
               (long long)workspace_bytes, (long long)need);
  FmBnArgs a{};
  a.col = col; a.B = B; a.F = (int)F; a.K = (int)K; a.V = V; a.bias = bias; a.b0 = b0; a.labels = labels; a.out = out;
  a.gV = gV; a.gbias = gbias; a.gb0 = gb0; a.loss_partials = loss_partials;
  a.touch_stamp = touch_stamp; a.stamp = stamp; a.touched_rows = touched_rows; a.touched_count = touched_count;
  a.hot = HotPlan{hot_slot, ghot, ghot_bias, n_rep, n_hot};
  a.keep = keep; a.drop_seed = drop_seed;
  a.gamma = gamma; a.beta = beta; a.mm = moving_mean; a.mv = moving_var; a.dgamma = dgamma; a.dbeta = dbeta;
  a.eps = eps; a.decay = decay;
  fm_bn_ws_bind(a, workspace);
  const cudaStream_t st = (cudaStream_t)stream;
  if (keep < 1.f) {
#define CALL(L, Vp) return launch_fm_bn_train<L, Vp, true>(a, deterministic, st)
    HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  } else {
#define CALL(L, Vp) return launch_fm_bn_train<L, Vp, false>(a, deterministic, st)
    HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  }
  return HHFM_ERR_UNSUPPORTED;
}

extern "C" int64_t hhfm_workspace_bytes_fm_bn_sync(int64_t B, int64_t K) {
  if (B < 0 || K <= 0 || K > 512) return -1;
  return (int64_t)fm_bn_sync_ws_bytes(B, K);
}

extern "C" int64_t hhfm_fm_bn_sync_len(int64_t K) {
  if (K <= 0 || K > 512) return -1;
  return 2 * K + 1;
}

extern "C" int hhfm_fm_bn_sync_stats(const int32_t* col, int64_t B, int64_t F, const float* V, const float* bias, int64_t M,
                                     int64_t K, double* stats, void* workspace, int64_t workspace_bytes, hhfm_stream_t stream) {
  int rc = check_bn_sync("fm_bn_sync_stats", B, K, 1, 0, stats, workspace, workspace_bytes);
  if (rc) return rc;
  rc = check_bn_rows(B, F, B == 0 && col == nullptr ? (const void*)V : col, V, M, K);     // an empty rank may pass col = NULL
  if (rc) return rc;
  FmBnArgs a{};
  a.col = col; a.B = B; a.F = (int)F; a.K = (int)K; a.V = V; a.bias = bias;
  fm_bn_ws_bind(a, workspace, true);
#define CALL(L, Vp) return launch_fm_bn_sync_stats<L, Vp>(a, stats, (cudaStream_t)stream)
  HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  return HHFM_ERR_UNSUPPORTED;
}

extern "C" int hhfm_fm_bn_sync_loss(int64_t B, int64_t K, const float* b0, const float* labels, float* out, float* gb0,
                                    float* loss_partials, float keep, uint64_t drop_seed, const float* gamma, const float* beta,
                                    float* moving_mean, float* moving_var, float eps, float decay, const double* stats_all,
                                    int32_t n_ranks, int32_t rank, double* sums, void* workspace, int64_t workspace_bytes,
                                    hhfm_stream_t stream) {
  int rc = check_bn_sync("fm_bn_sync_loss", B, K, n_ranks, rank, stats_all, workspace, workspace_bytes);
  if (rc) return rc;
  rc = check_bn_layer(gamma, beta, moving_mean, moving_var, eps);
  if (rc) return rc;
  HHFM_REQUIRE(sums != nullptr && ((uintptr_t)sums & 7) == 0, "fm_bn_sync_loss: sums must be non-NULL and 8-byte aligned");
  HHFM_REQUIRE((labels || B == 0) && loss_partials, "fm_bn: labels and loss_partials are required");
  HHFM_REQUIRE(keep > 0.f && keep <= 1.f, "fm_bn: dropout keep must be in (0, 1]");
  HHFM_REQUIRE(decay >= 0.f && decay < 1.f, "fm_bn: decay must be in [0, 1) (got %g)", (double)decay);
  FmBnArgs a{};
  a.B = B; a.K = (int)K; a.b0 = b0; a.labels = labels; a.out = out; a.gb0 = gb0; a.loss_partials = loss_partials;
  a.keep = keep; a.drop_seed = drop_seed;
  a.gamma = gamma; a.beta = beta; a.mm = moving_mean; a.mv = moving_var; a.eps = eps; a.decay = decay;
  fm_bn_ws_bind(a, workspace, true);
  const cudaStream_t st = (cudaStream_t)stream;
  if (keep < 1.f) {
#define CALL(L, Vp) return launch_fm_bn_sync_loss<L, Vp, true>(a, stats_all, n_ranks, rank, sums, st)
    HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  } else {
#define CALL(L, Vp) return launch_fm_bn_sync_loss<L, Vp, false>(a, stats_all, n_ranks, rank, sums, st)
    HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  }
  return HHFM_ERR_UNSUPPORTED;
}

extern "C" int hhfm_fm_bn_sync_scatter(const int32_t* col, int64_t B, int64_t F, const float* V, int64_t M, int64_t K,
                                       float* gV, float* gbias, int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows,
                                       int32_t* touched_count, const int32_t* hot_slot, float* ghot, float* ghot_bias,
                                       int32_t n_rep, int32_t n_hot, int32_t deterministic, float keep, uint64_t drop_seed,
                                       float* dgamma, float* dbeta, const double* sums_all, int32_t n_ranks, void* workspace,
                                       int64_t workspace_bytes, hhfm_stream_t stream) {
  int rc = check_bn_sync("fm_bn_sync_scatter", B, K, n_ranks, 0, sums_all, workspace, workspace_bytes);
  if (rc) return rc;
  rc = check_bn_rows(B, F, B == 0 && col == nullptr ? (const void*)V : col, V, M, K);
  if (rc) return rc;
  HHFM_REQUIRE(gV != nullptr, "fm_bn: gV is required");
  HHFM_REQUIRE(dgamma && dbeta, "fm_bn: dgamma and dbeta must not be NULL");
  rc = check_bn_scatter(touch_stamp, touched_rows, touched_count, hot_slot, ghot, n_rep, n_hot, gV, keep);
  if (rc) return rc;
  FmBnArgs a{};
  a.col = col; a.B = B; a.F = (int)F; a.K = (int)K; a.V = V; a.gV = gV; a.gbias = gbias;
  a.touch_stamp = touch_stamp; a.stamp = stamp; a.touched_rows = touched_rows; a.touched_count = touched_count;
  a.hot = HotPlan{hot_slot, ghot, ghot_bias, n_rep, n_hot};
  a.keep = keep; a.drop_seed = drop_seed; a.dgamma = dgamma; a.dbeta = dbeta;
  fm_bn_ws_bind(a, workspace, true);
  const cudaStream_t st = (cudaStream_t)stream;
  if (keep < 1.f) {
#define CALL(L, Vp) return launch_fm_bn_sync_scatter<L, Vp, true>(a, sums_all, n_ranks, deterministic, st)
    HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  } else {
#define CALL(L, Vp) return launch_fm_bn_sync_scatter<L, Vp, false>(a, sums_all, n_ranks, deterministic, st)
    HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  }
  return HHFM_ERR_UNSUPPORTED;
}

extern "C" int hhfm_fm_bn_fwd(const int32_t* col, int64_t B, int64_t F, const float* V, const float* bias, const float* b0,
                              int64_t M, int64_t K, const float* gamma, const float* beta, const float* moving_mean,
                              const float* moving_var, float eps, float* out, hhfm_stream_t stream) {
  int rc = check_bn_common(B, F, col, V, M, K, gamma, beta, moving_mean, moving_var, eps);
  if (rc) return rc;
  HHFM_REQUIRE(out != nullptr, "fm_bn_fwd: out is NULL");
  if (B == 0) return HHFM_OK;
  FmBnArgs a{};
  a.col = col; a.B = B; a.F = (int)F; a.K = (int)K; a.V = V; a.bias = bias; a.b0 = b0; a.out = out;
  a.gamma = gamma; a.beta = beta; a.mm = const_cast<float*>(moving_mean); a.mv = const_cast<float*>(moving_var); a.eps = eps;
#define CALL(L, Vp) return launch_fm_bn_fwd<L, Vp>(a, (cudaStream_t)stream)
  HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  return HHFM_ERR_UNSUPPORTED;
}
