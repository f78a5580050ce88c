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
};

static inline size_t bn_align(size_t b) { return (b + 255) / 256 * 256; }

static size_t fm_bn_ws_bytes(int64_t B, int64_t K) {
  return bn_align((size_t)B * K * 4) + 2 * bn_align((size_t)B * 4) + bn_align((size_t)kPartials * (2 * K + 1) * 4) +
         bn_align((size_t)5 * K * 4);
}

static void fm_bn_ws_bind(FmBnArgs& a, void* ws) {
  char* p = static_cast<char*>(ws);
  a.x = reinterpret_cast<float*>(p);     p += bn_align((size_t)a.B * a.K * 4);
  a.bsum = reinterpret_cast<float*>(p);  p += bn_align((size_t)a.B * 4);
  a.g = reinterpret_cast<float*>(p);     p += bn_align((size_t)a.B * 4);
  a.part = reinterpret_cast<float*>(p);  p += bn_align((size_t)kPartials * (2 * a.K + 1) * 4);
  a.colv = reinterpret_cast<float*>(p);
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
        m.v[i] = bn_mask(a, valid ? s : 0, 4 * (lg + i * LPS));
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
// of a column are merged in segment order by the thread of segment 0.
constexpr int kReduceThreads = 1024;     // one CTA does the whole merge: more threads, fewer partials each

template <bool STATS>
__global__ void __launch_bounds__(kReduceThreads) fm_bn_reduce_kernel(const FmBnArgs a, int n_part) {
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
          const double nb = q[2 * K];
          if (nb == 0.0) continue;
          const double nn = r0 + nb, d = (double)q[c] - r1;
          r1 += d * (nb / nn);
          r2 += (double)q[K + c] + d * d * (r0 * nb / nn);
          r0 = nn;
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
          const double nb = sh[0][o];
          if (nb == 0.0) continue;
          const double nn = r0 + nb, d = sh[1][o] - r1;
          r1 += d * (nb / nn);
          r2 += sh[2][o] + d * d * (r0 * nb / nn);
          r0 = nn;
        } else {
          r0 += sh[0][o];
          r1 += sh[1][o];
        }
      }
      if (STATS) {
        // normalisation: biased batch variance; moving variance: Bessel-corrected, B - 1 taken as 1 when B = 1 (the fused
        // batch-norm kernel of tf.contrib.layers.batch_norm, DESIGN.md 7)
        const float mu = (float)r1, var = (float)(r2 / (double)a.B);
        const float var_u = (float)(r2 / (double)(a.B > 1 ? a.B - 1 : 1));
        const float is = 1.f / sqrtf(var + a.eps);
        const float f = 1.f - a.decay;
        a.mm[c] = a.mm[c] - (a.mm[c] - mu) * f;
        a.mv[c] = a.mv[c] - (a.mv[c] - var_u) * f;
        a.colv[c] = mu;
        a.colv[K + c] = is;
        a.colv[2 * K + c] = a.gamma[c] * is;
      } else {
        const float db = (float)r0, dg = (float)r1;
        a.dbeta[c] = db;
        a.dgamma[c] = dg;
        a.colv[3 * K + c] = db / (float)a.B;
        a.colv[4 * K + c] = dg / (float)a.B;
      }
    }
    __syncthreads();
  }
  if (!STATS && threadIdx.x == 0 && a.gb0 != nullptr) {
    double t = 0.0;
    for (int p = 0; p < n_part; p++) t += a.part[(size_t)p * W + 2 * K];
    *a.gb0 += (float)t;
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
        const float4 d = DROP ? f4_mul(make_float4(g, g, g, g), f4_div(bn_mask(a, s, 4 * c), a.keep)) : make_float4(g, g, g, g);
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

template <int LPS, int VPL, bool DROP>
static int launch_fm_bn_train(FmBnArgs a, int deterministic, cudaStream_t st) {
  static int g1 = 0, g3 = 0, g5 = 0;          // CTAs per SM of each pass (the grid is this times the SMs, capped by B)
  if (g1 == 0) {
    g1 = bn_grid(fm_bn_gather_kernel<LPS, VPL>, (int64_t)1 << 40, LPS);
    g3 = bn_grid(fm_bn_loss_kernel<LPS, VPL, DROP>, (int64_t)1 << 40, LPS);
    g5 = bn_grid(fm_bn_scatter_kernel<LPS, VPL, DROP>, (int64_t)1 << 40, LPS);
  }
  const int64_t per_cta = (kBlock / 32) * (32 / LPS);
  auto grid = [&](int cap) { const int64_t need = (a.B + per_cta - 1) / per_cta; return (int)(need < cap ? need : cap); };
  const int n1 = grid(g1), n3 = grid(g3);
  fm_bn_gather_kernel<LPS, VPL><<<n1, kBlock, 0, st>>>(a);
  fm_bn_reduce_kernel<true><<<1, kReduceThreads, 0, st>>>(a, n1);
  fm_bn_loss_kernel<LPS, VPL, DROP><<<n3, kBlock, 0, st>>>(a);
  fm_bn_reduce_kernel<false><<<1, kReduceThreads, 0, st>>>(a, n3);
  if (deterministic) {                          // one warp in program order: bit-reproducible row gradients
    a.groups_active = 1;
    fm_bn_scatter_kernel<LPS, VPL, DROP><<<1, 32, 0, st>>>(a);
  } else {
    a.groups_active = 32 / LPS;
    fm_bn_scatter_kernel<LPS, VPL, DROP><<<grid(g5), kBlock, 0, st>>>(a);
  }
  return check_launch("fm_bn training kernels");
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

static int check_bn_common(int64_t B, int64_t F, const void* col, const void* V, int64_t M, int64_t K, const float* gamma,
                           const float* beta, const float* mm, const float* mv, float eps) {
  HHFM_REQUIRE(B >= 0 && M > 0, "fm_bn: bad sizes B=%lld M=%lld", (long long)B, (long long)M);
  HHFM_REQUIRE(col != nullptr && V != nullptr, "fm_bn: col and V must not be NULL");
  HHFM_REQUIRE(K > 0 && K % 4 == 0 && K <= 512, "fm_bn: K=%lld unsupported (need K %% 4 == 0, K <= 512)", (long long)K);
  HHFM_REQUIRE(F > 0, "fm_bn: F=%lld, need F > 0", (long long)F);
  HHFM_REQUIRE(gamma && beta && mm && mv, "fm_bn: gamma, beta, moving_mean and moving_var must not be NULL");
  HHFM_REQUIRE(((uintptr_t)V & 15) == 0, "fm_bn: V must be 16-byte aligned");
  HHFM_REQUIRE((((uintptr_t)gamma | (uintptr_t)beta | (uintptr_t)mm | (uintptr_t)mv) & 15) == 0,
               "fm_bn: gamma, beta, moving_mean and moving_var must be 16-byte aligned");
  HHFM_REQUIRE(eps > 0.f && eps < INFINITY, "fm_bn: eps must be > 0 (got %g)", (double)eps);
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
  HHFM_REQUIRE(!hot_slot || (ghot && n_rep >= 1 && n_hot >= 1), "fm_bn: hot_slot needs ghot, n_rep, n_hot");
  HHFM_REQUIRE(!touch_stamp || (touched_rows && touched_count), "fm_bn: touch_stamp needs touched_rows/count");
  HHFM_REQUIRE(((uintptr_t)gV & 15) == 0, "fm_bn: gV must be 16-byte aligned");
  HHFM_REQUIRE(keep > 0.f && keep <= 1.f, "fm_bn: dropout keep must be in (0, 1]");
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
