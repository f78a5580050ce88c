// K8: DeepFM (Newcode/DFM.py:104-152), fp32.
//
//   E = V[x] [F,K];  y1_f = feature_bias[x_f];  y2 = 0.5((sum_f e_f)^2 - sum_f e_f^2)            (DFM.py:104-122)
//   H_0 = reshape(E) [F*K];  H_i = relu(H_{i-1} W_{i-1} + b_{i-1}),  i = 1..L                     (DFM.py:125-128)
//   out = [y1 | y2 | H_L] . proj + cbias;  loss = 0.5 sum (y - out)^2  (+ l2 through the optimizer)   (DFM.py:131-152)
//
// The reference's options select parts of this graph independently (hhfm_dfm_mode bits): use_fm=False drops y1 / y2,
// use_deep=False drops the tower (out = [y1 | y2] . proj + cbias), loss_type='logloss' makes out = sigmoid(logit) and the loss
// tf.losses.log_loss(y, out) = mean_s [-y log(out + 1e-7) - (1 - y) log((1 - out) + 1e-7)].
//
// Two kernels:
//  * `sgemm_kernel<AMODE,BMODE,EPI>`: a 128x64x16 register-blocked fp32 SIMT GEMM (8x4 outputs per thread, double-
//    buffered shared tiles) whose A operand can be GATHERED from the embedding table (layer 0 never materialises
//    the [B, F*K] activation in HBM), whose epilogue fuses bias+relu, the relu mask of the backward (+ the bias
//    gradient column sums), split-K atomics for weight gradients, or the SCATTER of d(H_0) straight into the
//    embedding-gradient rows (sort-free vector reductions).  fp32 on CUDA cores because the parity bar is 1e-5
//    relative: tcgen05 has no fp32-input MMA kind (a 3xTF32 split is the planned faster variant).
//  * `dfm_head_kernel<VPL,TRAIN>`: one warp per sample: FM part, projection, loss, d(out), dZ_L, FM-part scatter and
//    the projection / last-bias gradients.
//
// Parameter block (one flat caller-owned buffer, gradients use the same layout):
//   [ layer_0 (d0 x d1) | ... | layer_{L-1} (d_{L-1} x d_L) | concat_projection (F+K+d_L) |   <- l2-regularised part
//     bias_0 (d1) | ... | bias_{L-1} (d_L) | concat_bias (1) ]
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "dfm_tc.cuh"

namespace hhfm {

enum { A_ROW = 0, A_COL = 1, A_GATHER = 2, A_GATHER_T = 3 };
enum { B_ROW = 0, B_COL = 1 };
enum { EPI_STORE = 0, EPI_BIAS_RELU = 1, EPI_MASK = 2, EPI_ATOMIC = 3, EPI_SCATTER = 4 };

constexpr int BM = 128, BN = 64, BK = 16;
constexpr int LDAS = BM + 4, LDBS = BN + 4;
constexpr int kDfmMaxLayers = 8;

struct GemmArgs {
  const float* A;        // dense operand, or the embedding table V in the gather modes
  const float* B;
  float* C;
  int M, N, Kd;
  int64_t lda, ldb, ldc;
  const int32_t* idx;    // [rows, F] (gather modes, EPI_SCATTER)
  int F, K;
  const float* bias;     // EPI_BIAS_RELU: [N]
  const float* mask;     // EPI_MASK: C = acc * (mask > 0); may alias C
  int64_t ldmask;
  float* colsum;         // EPI_MASK, optional: colsum[n] += sum_m C[m,n]
  int k_chunk;           // split-K: blockIdx.z covers [z*k_chunk, (z+1)*k_chunk)
  HotPlan hot;           // EPI_SCATTER: optional hot-row replicas
};

// A-operand element (m, k).  In the gather modes (f, c) = (field, offset inside the embedding row) of the gathered
// coordinate are precomputed by the caller so the inner loads carry no integer division.
template <int AMODE>
__device__ __forceinline__ float load_a(const GemmArgs& g, int m, int k, int f, int c) {
  if (m >= g.M || k >= g.Kd) return 0.f;
  if (AMODE == A_ROW) return __ldg(g.A + (int64_t)m * g.lda + k);
  if (AMODE == A_COL) return __ldg(g.A + (int64_t)k * g.lda + m);
  const int sample = (AMODE == A_GATHER) ? m : k;
  const int row = __ldg(g.idx + (int64_t)sample * g.F + f);
  return __ldg(g.A + (int64_t)row * g.K + c);
}

template <int BMODE>
__device__ __forceinline__ float load_b(const GemmArgs& g, int k, int n) {
  if (n >= g.N || k >= g.Kd) return 0.f;
  if (BMODE == B_ROW) return __ldg(g.B + (int64_t)k * g.ldb + n);
  return __ldg(g.B + (int64_t)n * g.ldb + k);
}

template <int AMODE, int BMODE, int EPI>
__global__ void __launch_bounds__(256) sgemm_kernel(const GemmArgs g) {
  __shared__ __align__(16) float As[2][BK][LDAS];
  __shared__ __align__(16) float Bs[2][BK][LDBS];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  int k_beg = 0, k_end = g.Kd;
  if (EPI == EPI_ATOMIC) {
    k_beg = blockIdx.z * g.k_chunk;
    k_end = min(g.Kd, k_beg + g.k_chunk);
    if (k_beg >= k_end) return;
  }
  constexpr bool A_KC = (AMODE == A_ROW || AMODE == A_GATHER);   // k is the contiguous index of the A operand
  constexpr bool B_KC = (BMODE == B_COL);

  float ra[8], rb[4];
  int gf = 0, gc = 0;        // A_GATHER_T: (field, offset) of this thread's fixed m
  if (AMODE == A_GATHER_T) {
    const int m = m0 + (tid & 127);
    gf = m / g.K;
    gc = m - gf * g.K;
  }
  auto fetch = [&](int k0) {
    if (AMODE == A_GATHER) {   // (field, offset) of this thread's k = k0 + (tid & 15)
      gf = k0 / g.K;
      gc = k0 - gf * g.K + (tid & 15);
      while (gc >= g.K) { gc -= g.K; gf++; }
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int mm = A_KC ? ((tid >> 4) + 16 * i) : (tid & 127);
      const int kk = A_KC ? (tid & 15) : ((tid >> 7) + 2 * i);
      const int k = k0 + kk;
      ra[i] = (k < k_end) ? load_a<AMODE>(g, m0 + mm, k, gf, gc) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int nn = B_KC ? ((tid >> 4) + 16 * i) : (tid & 63);
      const int kk = B_KC ? (tid & 15) : ((tid >> 6) + 4 * i);
      const int k = k0 + kk;
      rb[i] = (k < k_end) ? load_b<BMODE>(g, k, n0 + nn) : 0.f;
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int mm = A_KC ? ((tid >> 4) + 16 * i) : (tid & 127);
      const int kk = A_KC ? (tid & 15) : ((tid >> 7) + 2 * i);
      As[buf][kk][mm] = ra[i];
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int nn = B_KC ? ((tid >> 4) + 16 * i) : (tid & 63);
      const int kk = B_KC ? (tid & 15) : ((tid >> 6) + 4 * i);
      Bs[buf][kk][nn] = rb[i];
    }
  };

  float acc[8][4];
#pragma unroll
  for (int r = 0; r < 8; r++)
#pragma unroll
    for (int c = 0; c < 4; c++) acc[r][c] = 0.f;

  fetch(k_beg);
  stash(0);
  __syncthreads();
  int buf = 0;
  for (int k0 = k_beg; k0 < k_end; k0 += BK) {
    const bool more = (k0 + BK) < k_end;
    if (more) fetch(k0 + BK);
#pragma unroll
    for (int kk = 0; kk < BK; kk++) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 8 + 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int r = 0; r < 8; r++)
#pragma unroll
        for (int c = 0; c < 4; c++) acc[r][c] = fmaf(av[r], bv[c], acc[r][c]);
    }
    if (more) {
      stash(buf ^ 1);
      __syncthreads();
      buf ^= 1;
    }
  }

  // ---- epilogue ----
  const int nb = n0 + tx * 4;
  float cs[4] = {0.f, 0.f, 0.f, 0.f};
  const int sf = (EPI == EPI_SCATTER) ? nb / g.K : 0;
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const int m = m0 + ty * 8 + r;
    if (m >= g.M) continue;
    if (EPI == EPI_SCATTER) {
      // d(H_0)[m, n] belongs to embedding row idx[m, n / K], element n % K; 4 consecutive n share a row (K % 4 == 0)
      if (nb < g.N) {
        const int row = __ldg(g.idx + (int64_t)m * g.F + sf);
        float* dstrow = g.C + (int64_t)row * g.K;
        if (g.hot.slot) {
          const int hs = __ldg(g.hot.slot + row);
          if (hs >= 0) dstrow = g.hot.ghot + ((size_t)(blockIdx.x % g.hot.n_rep) * g.hot.n_hot + hs) * g.K;
        }
        red_add_v4(dstrow + (nb - sf * g.K), make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]));
      }
      continue;
    }
#pragma unroll
    for (int c = 0; c < 4; c++) {
      const int n = nb + c;
      if (n >= g.N) continue;
      float v = acc[r][c];
      float* dst = g.C + (int64_t)m * g.ldc + n;
      if (EPI == EPI_BIAS_RELU) v = fmaxf(v + __ldg(g.bias + n), 0.f);
      if (EPI == EPI_MASK) {
        v = (g.mask[(int64_t)m * g.ldmask + n] > 0.f) ? v : 0.f;
        cs[c] += v;
      }
      if (EPI == EPI_ATOMIC) atomicAdd(dst, v);
      else *dst = v;
    }
  }
  if (EPI == EPI_MASK && g.colsum != nullptr) {
    // bias gradient: column sums of this tile (16 row-groups -> shared -> one atomic per column)
    __syncthreads();
    float* red = &As[0][0][0];     // 16 x 64 floats
#pragma unroll
    for (int c = 0; c < 4; c++) red[ty * BN + tx * 4 + c] = cs[c];
    __syncthreads();
    if (tid < BN && n0 + tid < g.N) {
      float s = 0.f;
#pragma unroll
      for (int r = 0; r < 16; r++) s += red[r * BN + tid];
      atomicAdd(g.colsum + n0 + tid, s);
    }
  }
}

template <int AMODE, int BMODE, int EPI>
static int launch_gemm(GemmArgs g, cudaStream_t st) {
  if (g.M <= 0 || g.N <= 0 || g.Kd <= 0) return HHFM_OK;
  dim3 grid((g.M + BM - 1) / BM, (g.N + BN - 1) / BN, 1);
  if (EPI == EPI_ATOMIC) {
    const int64_t tiles = (int64_t)grid.x * grid.y;
    int64_t splits = (4 * (int64_t)sm_count() + tiles - 1) / tiles;
    const int64_t max_splits = (g.Kd + 8 * BK - 1) / (8 * BK);
    if (splits > max_splits) splits = max_splits;
    if (splits < 1) splits = 1;
    int64_t chunk = (g.Kd + splits - 1) / splits;
    chunk = (chunk + BK - 1) / BK * BK;
    g.k_chunk = (int)chunk;
    grid.z = (unsigned)((g.Kd + chunk - 1) / chunk);
  }
  sgemm_kernel<AMODE, BMODE, EPI><<<grid, 256, 0, st>>>(g);
  return check_launch("sgemm_kernel");
}

// --------------------------------------------------------------------------------------------------------------
struct HeadArgs {
  const int32_t* idx;
  int64_t B;
  int F, K, D;             // D = width of the last hidden layer
  const float* V;
  const float* fbias;      // feature_bias [M]
  const float* proj;       // [F + K + D]
  const float* cbias;      // [1]
  float* H;                // [B, ldh]: H_L on entry; dZ_L on exit (TRAIN)
  int64_t ldh;
  const float* labels;
  float* out;
  float* gV;
  float* gfbias;
  float* gproj;            // [F + K + D]
  float* gcbias;           // [1]
  float* gblast;           // [D]  bias gradient of the last hidden layer = column sums of dZ_L
  float* loss_partials;
  HotPlan hot;             // optional hot-row replicas for the FM-part scatter
  int fm;                  // 1: first- and second-order terms (and their gradients); 0: out = H_L . proj3 + cbias (+ extra)
  int loss;                // HEAD_SQ / HEAD_WD / HEAD_LOGLOSS (HEAD_LOGLOSS: out[s] = sigmoid(logit))
  // Wide&Deep (WDMF.py:51-126): no FM terms, out = H_L . proj3 + cbias + extra[s] is a logit, loss = mean sigmoid
  // cross-entropy over the batch, d loss / d out is also written per sample for the wide part's scatter
  const float* extra;      // [B] additive logit (the wide part) or NULL
  float* gsample;          // [B] d loss / d out (TRAIN) or NULL
  float inv_b;             // 1 / B (WD), 1 / B_total (log_loss: the batch the mean runs over, all ranks together)
};

// loss heads: 0.5 (y - out)^2 summed (DeepFM mse); WD's mean sigmoid cross-entropy on the logit; DeepFM's
// tf.losses.log_loss on the sigmoid (DFM.py:139-141), TF's epsilon and evaluation order
enum { HEAD_SQ = 0, HEAD_WD = 1, HEAD_LOGLOSS = 2 };
constexpr float kLogLossEps = 1e-7f;

constexpr int kHeadT = 8;    // D <= 32 * kHeadT

// LOG: the log_loss head (a.loss == HEAD_LOGLOSS) as its own instance, so the other heads keep their register budget
template <int VPL, bool TRAIN, bool LOG>
__global__ void __launch_bounds__(256) dfm_head_kernel(const HeadArgs a) {
  extern __shared__ float sred[];         // TRAIN: [F + K + 2*D + 1]
  __shared__ float scratch[32];
  const int lane = threadIdx.x & 31;
  const int F = a.F, K = a.K, D = a.D, kv = K >> 2;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int nred = F + K + 2 * D + 1;
  if (TRAIN) {
    for (int i = threadIdx.x; i < nred; i += blockDim.x) sred[i] = 0.f;
    __syncthreads();
  }
  const float cb = __ldg(a.cbias);
  const float p1 = (lane < F) ? __ldg(a.proj + lane) : 0.f;
  float4 p2[VPL];
#pragma unroll
  for (int i = 0; i < VPL; i++) {
    const int c = lane + 32 * i;
    const float* q = a.proj + F + 4 * c;            // the projection block has no 16-byte alignment guarantee
    p2[i] = (c < kv) ? make_float4(__ldg(q), __ldg(q + 1), __ldg(q + 2), __ldg(q + 3)) : f4_zero();
  }
  float p3[kHeadT];
#pragma unroll
  for (int t = 0; t < kHeadT; t++) p3[t] = (lane + 32 * t < D) ? __ldg(a.proj + F + K + lane + 32 * t) : 0.f;

  const int rep = a.hot.slot ? (int)(warp_g % a.hot.n_rep) : 0;
  float g1 = 0.f, gcb = 0.f, loss_acc = 0.f;
  float4 g2[VPL];
  float g3[kHeadT], gbl[kHeadT];
#pragma unroll
  for (int i = 0; i < VPL; i++) g2[i] = f4_zero();
#pragma unroll
  for (int t = 0; t < kHeadT; t++) { g3[t] = 0.f; gbl[t] = 0.f; }

  for (int64_t s = warp_g; s < a.B; s += n_warps) {
    const int my_id = (lane < F && a.fm) ? __ldg(a.idx + s * F + lane) : 0;
    const float y1 = (lane < F && a.fm) ? __ldg(a.fbias + my_id) : 0.f;
    float4 S[VPL], Q[VPL];
#pragma unroll
    for (int i = 0; i < VPL; i++) { S[i] = f4_zero(); Q[i] = f4_zero(); }
    for (int f = 0; f < (a.fm ? F : 0); f++) {
      const int id = __shfl_sync(0xffffffffu, my_id, f);
      const float4* row = reinterpret_cast<const float4*>(a.V) + (size_t)id * kv;
#pragma unroll
      for (int i = 0; i < VPL; i++) {
        const int c = lane + 32 * i;
        if (c < kv) {
          const float4 e = ldg4(row + c);
          S[i] = f4_add(S[i], e);
          Q[i] = f4_add(Q[i], f4_mul(e, e));
        }
      }
    }
    float4 y2[VPL];
    float part = y1 * p1;
#pragma unroll
    for (int i = 0; i < VPL; i++) {
      y2[i] = f4_scale(f4_sub(f4_mul(S[i], S[i]), Q[i]), 0.5f);
      part += f4_dot(y2[i], p2[i]);
    }
    float h[kHeadT];
    float* hrow = a.H + s * a.ldh;
#pragma unroll
    for (int t = 0; t < kHeadT; t++) {
      const int j = lane + 32 * t;
      h[t] = (j < D) ? hrow[j] : 0.f;
      part = fmaf(h[t], p3[t], part);
    }
    float out = warp_sum(part) + cb;
    if (a.loss == HEAD_WD && a.extra) out += __ldg(a.extra + s);
    const float pr = LOG ? 1.f / (1.f + expf(-out)) : out;
    if (lane == 0 && a.out) a.out[s] = pr;
    if (!TRAIN) continue;

    float g;
    if (LOG) {
      // per sample -y log(p + eps) - (1 - y) log((1 - p) + eps), mean over B_total; d/d logit = p (1 - p) d/dp (TF's
      // SigmoidGrad).  Labels are used as given (the drop-in trainer's negatives are -1).
      const float y = __ldg(a.labels + s);
      const float q = 1.f - pr;
      loss_acc += (lane == 0) ? (-(y * logf(pr + kLogLossEps)) - (1.f - y) * logf(q + kLogLossEps)) * a.inv_b : 0.f;
      const float dp = (-y / (pr + kLogLossEps) + (1.f - y) / (q + kLogLossEps)) * a.inv_b;
      g = dp * pr * q;
    } else if (a.loss == HEAD_WD) {
      // mean sigmoid cross-entropy, labels in {0, 1}: loss = (max(z,0) - z y + log(1 + exp(-|z|))) / B, d/dz = (sigmoid(z) - y) / B
      const float y = __ldg(a.labels + s);
      const float pr = 1.f / (1.f + expf(-out));
      g = (pr - y) * a.inv_b;
      loss_acc += (lane == 0) ? (fmaxf(out, 0.f) - out * y + log1pf(expf(-fabsf(out)))) * a.inv_b : 0.f;
      if (lane == 0 && a.gsample) a.gsample[s] = g;
    } else {
      g = out - __ldg(a.labels + s);                  // d loss / d out, loss = 0.5 (y - out)^2
      loss_acc += (lane == 0) ? 0.5f * g * g : 0.f;
    }
    gcb += (lane == 0) ? g : 0.f;
    g1 = fmaf(g, y1, g1);
#pragma unroll
    for (int i = 0; i < VPL; i++) g2[i] = f4_fma(y2[i], g, g2[i]);
#pragma unroll
    for (int t = 0; t < kHeadT; t++) {
      const int j = lane + 32 * t;
      g3[t] = fmaf(g, h[t], g3[t]);
      const float dz = (h[t] > 0.f) ? g * p3[t] : 0.f;
      gbl[t] += dz;
      if (j < D) hrow[j] = dz;
    }
    if (!a.fm) continue;
    // FM part of the embedding gradient: dV[x_f] += g * proj2 * (S - e_f);  d feature_bias[x_f] += g * proj1[f]
    const int my_slot = (a.hot.slot && lane < F) ? __ldg(a.hot.slot + my_id) : -1;
    if (lane < F) {
      float* pb = a.gfbias + my_id;
      if (my_slot >= 0 && a.hot.ghot_bias != nullptr) pb = a.hot.ghot_bias + (size_t)rep * a.hot.n_hot + my_slot;
      atomicAdd(pb, g * p1);
    }
    for (int f = 0; f < F; f++) {
      const int id = __shfl_sync(0xffffffffu, my_id, f);
      const float4* row = reinterpret_cast<const float4*>(a.V) + (size_t)id * kv;
      const int slot = __shfl_sync(0xffffffffu, my_slot, f);
      float* dst = (slot >= 0) ? a.hot.ghot + ((size_t)rep * a.hot.n_hot + slot) * K : a.gV + (size_t)id * K;
#pragma unroll
      for (int i = 0; i < VPL; i++) {
        const int c = lane + 32 * i;
        if (c < kv) {
          const float4 e = ldg4(row + c);
          red_add_v4(dst + 4 * c, f4_scale(f4_mul(p2[i], f4_sub(S[i], e)), g));
        }
      }
    }
  }
  if (!TRAIN) return;
  // ---- CTA reduction of the small dense gradients, then one global atomic per element ----
  if (lane < F) atomicAdd(&sred[lane], g1);
#pragma unroll
  for (int i = 0; i < VPL; i++) {
    const int c = lane + 32 * i;
    if (c < kv) {
      atomicAdd(&sred[F + 4 * c + 0], g2[i].x);
      atomicAdd(&sred[F + 4 * c + 1], g2[i].y);
      atomicAdd(&sred[F + 4 * c + 2], g2[i].z);
      atomicAdd(&sred[F + 4 * c + 3], g2[i].w);
    }
  }
#pragma unroll
  for (int t = 0; t < kHeadT; t++) {
    const int j = lane + 32 * t;
    if (j < D) {
      atomicAdd(&sred[F + K + j], g3[t]);
      atomicAdd(&sred[F + K + D + j], gbl[t]);
    }
  }
  if (lane == 0) atomicAdd(&sred[F + K + 2 * D], gcb);
  __syncthreads();
  for (int i = threadIdx.x; i < nred; i += blockDim.x) {
    const float v = sred[i];
    if (i < F + K + D) atomicAdd(a.gproj + i, v);
    else if (i < F + K + 2 * D) atomicAdd(a.gblast + (i - F - K - D), v);
    else atomicAdd(a.gcbias, v);
  }
  const float bl = block_sum(loss_acc, scratch);
  write_partial(a.loss_partials, bl);
}

template <bool TRAIN, bool LOG>
static void launch_head_vpl(const HeadArgs& a, int grid, size_t smem, cudaStream_t st) {
  const int kv = a.K >> 2;
  if (kv <= 32) dfm_head_kernel<1, TRAIN, LOG><<<grid, 256, smem, st>>>(a);
  else if (kv <= 64) dfm_head_kernel<2, TRAIN, LOG><<<grid, 256, smem, st>>>(a);
  else dfm_head_kernel<4, TRAIN, LOG><<<grid, 256, smem, st>>>(a);
}

template <bool TRAIN>
static int launch_head(const HeadArgs& a, cudaStream_t st) {
  const int grid = grid_for(a.B, 8, 4);
  const size_t smem = TRAIN ? (size_t)(a.F + a.K + 2 * a.D + 1) * sizeof(float) : 0;
  if (a.loss == HEAD_LOGLOSS) launch_head_vpl<TRAIN, true>(a, grid, smem, st);
  else launch_head_vpl<TRAIN, false>(a, grid, smem, st);
  return check_launch("dfm_head_kernel");
}

// --------------------------------------------------------------------------------------------------------------
struct DfmLayout {
  int L;
  int d[kDfmMaxLayers + 1];          // d[0] = F*K, d[i] = layer_sizes[i-1]
  int64_t ld[kDfmMaxLayers + 1];     // leading dimension of the H_i workspace block (d[i] rounded up to 4)
  int64_t w_off[kDfmMaxLayers];      // offsets into the parameter block
  int64_t b_off[kDfmMaxLayers];
  int64_t proj_off, cbias_off, total, reg_len;
  int64_t h_off[kDfmMaxLayers + 1];  // offsets into the workspace (floats); h_off[0] unused
  int64_t ws_floats;
};

// Mode bits (hhfm_dfm_mode) plus one internal bit for the Wide&Deep head, which callers cannot pass
constexpr int32_t kDfmPublicBits = HHFM_DFM_NO_FM | HHFM_DFM_NO_DEEP | HHFM_DFM_LOGLOSS;
constexpr int32_t kDfmWd = 1 << 8;

static bool dfm_fm(int32_t mode) { return !(mode & HHFM_DFM_NO_FM); }
static bool dfm_deep(int32_t mode) { return !(mode & HHFM_DFM_NO_DEEP); }

static int dfm_check_mode(int32_t mode) {
  HHFM_REQUIRE((mode & ~kDfmPublicBits) == 0, "dfm: unknown mode bits 0x%x (known: NO_FM 1, NO_DEEP 2, LOGLOSS 4)",
               (unsigned)(mode & ~kDfmPublicBits));
  HHFM_REQUIRE(dfm_fm(mode) || dfm_deep(mode), "dfm: mode %d enables neither the FM part nor the tower", (int)mode);
  return HHFM_OK;
}

static void dfm_head_mode(int32_t mode, HeadArgs& h) {
  h.fm = dfm_fm(mode) ? 1 : 0;
  h.loss = (mode & kDfmWd) ? HEAD_WD : (mode & HHFM_DFM_LOGLOSS) ? HEAD_LOGLOSS : HEAD_SQ;
}

// use_deep=False: the layer matrices keep their place (the model still owns them), the projection starts on a 16-byte
// boundary so the optimizer can step [proj_off, reg_len) alone, and no activation workspace is needed
static int dfm_layout(int64_t B, int64_t F, int64_t K, int32_t L, const int32_t* sizes, DfmLayout& lo, int32_t mode = 0) {
  HHFM_REQUIRE(L >= 1 && L <= kDfmMaxLayers && sizes, "dfm: 1 <= n_layers <= %d", kDfmMaxLayers);
  HHFM_REQUIRE(F >= 1 && F <= 32, "dfm: 1 <= field_size <= 32");
  HHFM_REQUIRE(K % 4 == 0 && K > 0 && K <= 512, "dfm: embedding_size must be a multiple of 4, <= 512");
  lo.L = L;
  lo.d[0] = (int)(F * K);
  int64_t off = 0, ws = 0;
  for (int i = 0; i < L; i++) {
    HHFM_REQUIRE(sizes[i] >= 1 && sizes[i] <= 4096, "dfm: layer size out of range");
    lo.d[i + 1] = sizes[i];
    lo.w_off[i] = off;
    off += (int64_t)lo.d[i] * lo.d[i + 1];
  }
  HHFM_REQUIRE(lo.d[L] <= 32 * kHeadT, "dfm: last hidden layer must be <= %d wide", 32 * kHeadT);
  if (!dfm_deep(mode)) off = (off + 3) / 4 * 4;
  lo.proj_off = off;
  off += F + K + lo.d[L];
  off = (off + 3) / 4 * 4;          // zero padding keeps the un-regularised tail 16-byte aligned for the optimizer
  lo.reg_len = off;
  for (int i = 0; i < L; i++) {
    lo.b_off[i] = off;
    off += lo.d[i + 1];
  }
  lo.cbias_off = off;
  lo.total = off + 1;
  for (int i = 1; i <= L; i++) {
    lo.ld[i] = (lo.d[i] + 3) / 4 * 4;
    lo.h_off[i] = ws;
    ws += B * lo.ld[i];
  }
  lo.ws_floats = dfm_deep(mode) ? ws : 0;
  return HHFM_OK;
}

// first > 0: H_first is already in the workspace (item-separable evaluator)
static int dfm_forward(const int32_t* idx, int64_t B, int64_t F, const float* V, int64_t K, const float* params,
                       const DfmLayout& lo, float* ws, cudaStream_t st, int first = 0) {
  for (int i = first; i < lo.L; i++) {
    GemmArgs g{};
    g.M = (int)B; g.N = lo.d[i + 1]; g.Kd = lo.d[i];
    g.B = params + lo.w_off[i]; g.ldb = lo.d[i + 1];
    g.C = ws + lo.h_off[i + 1]; g.ldc = lo.ld[i + 1];
    g.bias = params + lo.b_off[i];
    int rc;
    if (i == 0) {
      g.A = V; g.idx = idx; g.F = (int)F; g.K = (int)K;
      rc = launch_gemm<A_GATHER, B_ROW, EPI_BIAS_RELU>(g, st);
    } else {
      g.A = ws + lo.h_off[i]; g.lda = lo.ld[i];
      rc = launch_gemm<A_ROW, B_ROW, EPI_BIAS_RELU>(g, st);
    }
    if (rc != HHFM_OK) return rc;
  }
  return HHFM_OK;
}

// C[M,N] += A[Kd,M]^T B[Kd,N] (split over Kd, atomics): the shared fp32 CUDA-core GEMM for the small products of other models
int sgemm_tn_splitk(const float* A, int64_t lda, const float* B, int64_t ldb, int M, int N, int Kd, float* C, int64_t ldc,
                    cudaStream_t st) {
  GemmArgs g{};
  g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc; g.M = M; g.N = N; g.Kd = Kd;
  return launch_gemm<A_COL, B_ROW, EPI_ATOMIC>(g, st);
}

// ---- tensor-core path (dfm_tc.cu): every activation tensor X_l (l = 0: flattened embeddings, l >= 1: H_l, later dZ_l)
// lives in four forms: X [B, ld_l], X_lo, and the k-blocked transposes X^T / X^T_lo ([B/32 panels][d_l][32]); every layer matrix in padded forms W [d_i, ldp_i] (+lo)
// and W^T [d_{i+1}, ldt_i] (+lo).
struct DfmTcLayout {
  int64_t ldB;
  int64_t x[kDfmMaxLayers + 1], xlo[kDfmMaxLayers + 1], xt[kDfmMaxLayers + 1], xtlo[kDfmMaxLayers + 1];
  int64_t ldx[kDfmMaxLayers + 1];
  int64_t w[kDfmMaxLayers], wlo[kDfmMaxLayers], wt[kDfmMaxLayers], wtlo[kDfmMaxLayers];
  int ldp[kDfmMaxLayers], ldt[kDfmMaxLayers];
  int64_t scratch, scratch_floats;      // split-K partial tiles of the weight-gradient GEMMs
  int64_t total;
};

static bool dfm_use_tc(int64_t K) {
  const char* e = getenv("HHFM_DFM_TC");       // 0 = fp32 CUDA-core GEMMs, unset/1 = 3xTF32 tensor-core GEMMs
  if (e && e[0] == '0') return false;
  return K % 16 == 0;                          // the scatter epilogue maps 16-column chunks to one embedding row
}

// forward_from > 0: inference that enters at layer `forward_from` (the item-separable evaluator): no input forms below it
// and no transposed forms at all
static void dfm_tc_layout(int64_t B, const DfmLayout& lo, DfmTcLayout& t, int forward_from = 0) {
  auto r4 = [](int64_t x) { return (x + 3) / 4 * 4; };
  t.ldB = (B + 31) / 32 * 32;          // the transposed forms are k-blocked panels of 32 samples
  int64_t o = 0;
  for (int l = 0; l <= lo.L; l++) {
    t.ldx[l] = r4(lo.d[l]);
    const bool have = l >= forward_from;
    t.x[l] = o; o += have ? B * t.ldx[l] : 0;
    t.xlo[l] = o; o += have ? B * t.ldx[l] : 0;
    t.xt[l] = o; o += forward_from ? 0 : (int64_t)lo.d[l] * t.ldB;
    t.xtlo[l] = o; o += forward_from ? 0 : (int64_t)lo.d[l] * t.ldB;
  }
  for (int i = 0; i < lo.L; i++) {
    t.ldp[i] = (int)r4(lo.d[i + 1]);
    t.ldt[i] = (int)r4(lo.d[i]);
    t.w[i] = o; o += (int64_t)lo.d[i] * t.ldp[i];
    t.wlo[i] = o; o += (int64_t)lo.d[i] * t.ldp[i];
    t.wt[i] = o; o += (int64_t)lo.d[i + 1] * t.ldt[i];
    t.wtlo[i] = o; o += (int64_t)lo.d[i + 1] * t.ldt[i];
  }
  t.scratch = r4(o);
  t.scratch_floats = tf_splitk_scratch_floats();
  t.total = t.scratch + t.scratch_floats;
}

// first > 0 (inference only): X_first is already in the workspace (item-separable evaluator); its lo half is made here
static int dfm_tc_forward(const int32_t* idx, int64_t B, int64_t F, const float* V, int64_t K, const float* params,
                          const DfmLayout& lo, const DfmTcLayout& t, float* ws, bool train, cudaStream_t st, int first = 0,
                          bool first_has_lo = false, const float* proj_last = nullptr) {
  int rc;
  for (int i = first; i < lo.L; i++)
    if ((rc = tf_prep_weight(params + lo.w_off[i], lo.d[i], lo.d[i + 1], ws + t.w[i], ws + t.wlo[i], t.ldp[i], ws + t.wt[i],
                             ws + t.wtlo[i], t.ldt[i], st)))
      return rc;
  if (first == 0) {
    if ((rc = tf_gather_split_transpose(idx, B, (int)F, (int)K, V, ws + t.x[0], t.ldx[0], ws + t.xlo[0], train ? ws + t.xt[0] : nullptr,
                                        train ? ws + t.xtlo[0] : nullptr, st)))
      return rc;
  } else if (first < lo.L && !first_has_lo) {
    if ((rc = tf_split_transpose(ws + t.x[first], B, lo.d[first], t.ldx[first], ws + t.xlo[first], nullptr, nullptr, st))) return rc;
  }
  for (int i = first; i < lo.L; i++) {
    TfGemm g{};
    g.A = ws + t.x[i]; g.A_lo = ws + t.xlo[i]; g.lda = t.ldx[i];
    g.B = ws + t.wt[i]; g.B_lo = ws + t.wtlo[i]; g.ldb = t.ldt[i];
    g.M = (int)B; g.N = lo.d[i + 1]; g.K = lo.d[i];
    g.epi = TF_EPI_BIAS_RELU; g.C = ws + t.x[i + 1]; g.ldc = t.ldx[i + 1]; g.bias = params + lo.b_off[i];
    if (proj_last != nullptr && i == lo.L - 1) {
      // evaluator: the last hidden layer is only ever multiplied by the projection -- keep relu(H W + b) . proj as
      // tf_proj_partials() partial sums per row in the H_L block instead of writing and re-reading H_L
      g.epi = TF_EPI_BIAS_RELU_PROJ; g.proj = proj_last;
    }
    if ((rc = tf_gemm(g, st))) return rc;
    if (i + 1 < lo.L) {   // H_L is consumed by the head kernel as is (and replaced by dZ_L, split afterwards)
      const bool need_t = train;
      if ((rc = tf_split_transpose(ws + t.x[i + 1], B, lo.d[i + 1], t.ldx[i + 1], ws + t.xlo[i + 1],
                                   need_t ? ws + t.xt[i + 1] : nullptr, need_t ? ws + t.xtlo[i + 1] : nullptr, st)))
        return rc;
    }
  }
  return HHFM_OK;
}

// --------------------------------------------------------------------------------------------------------------
// Item-separable full-catalog evaluator (DFM.py:219-231; SURVEY 8f-3).  A context row with field item_col replaced by item n:
//   first hidden layer   Z1[c, n] = (b1 + sum_{f != item} E_cf W1_f) + E_n W1_item = U[c] + T[n]   (W1_f = rows f*K..(f+1)*K of W1)
//   first order          sum_{f != item} w[x_cf] proj[f]  +  w[n] proj[item_col]
//   second order         0.5 ((S_c + v_n)^2 - (Q_c + v_n^2)) . proj2,  S_c / Q_c = sums of E_cf / E_cf^2 over the context fields
// so the [F*K x d1] product (61 % of the tower's flops at 640-150-200-150), the 2.5 KB row gather and its tf32 split are
// paid once per context and once per item instead of once per (context, item).  Rows are ordered s = c * N + n.
// --------------------------------------------------------------------------------------------------------------
struct DfmTopnArgs {
  const int32_t* rows;
  int64_t row_stride;
  int C, F, K, item_col, d1;
  int64_t ld1;
  const float *V, *fbias, *W1, *b1, *proj;
  int64_t item_base, N;
  float *U, *T, *SQ, *fo;      // [C, ld1], [N, ld1] (tower only), [C, 2K], [C] (FM part only)
  int fm, deep, sig;           // parts of the graph the mode keeps; sig: scores are sigmoid(logit)
};

__global__ void __launch_bounds__(256) dfm_topn_ctx_kernel(const DfmTopnArgs a) {
  extern __shared__ float sE[];            // [F][K], the item field zeroed
  __shared__ float scratch[32];
  const int c = blockIdx.x, F = a.F, K = a.K;
  const int32_t* rec = a.rows + (int64_t)c * a.row_stride;
  for (int i = threadIdx.x; i < F * K; i += blockDim.x) {
    const int f = i / K, k = i % K;
    sE[i] = (f == a.item_col) ? 0.f : __ldg(a.V + (size_t)__ldg(rec + f) * K + k);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < (a.fm ? K : 0); k += blockDim.x) {
    float S = 0.f, Q = 0.f;
    for (int f = 0; f < F; f++) { const float e = sE[f * K + k]; S += e; Q = fmaf(e, e, Q); }
    a.SQ[(int64_t)c * 2 * K + k] = S;
    a.SQ[(int64_t)c * 2 * K + K + k] = Q;
  }
  if (a.fm) {
    float fo = 0.f;
    if ((int)threadIdx.x < F && (int)threadIdx.x != a.item_col) fo = __ldg(a.fbias + __ldg(rec + threadIdx.x)) * __ldg(a.proj + threadIdx.x);
    fo = block_sum(fo, scratch);
    if (threadIdx.x == 0) a.fo[c] = fo;
  }
  for (int j = threadIdx.x; j < (a.deep ? a.ld1 : 0); j += blockDim.x) {
    float acc = 0.f;
    if (j < a.d1) {
      for (int f = 0; f < F; f++) {
        if (f == a.item_col) continue;
        const float* w = a.W1 + (size_t)f * K * a.d1 + j;
        for (int k = 0; k < K; k++) acc = fmaf(sE[f * K + k], __ldg(w + (size_t)k * a.d1), acc);
      }
      acc += __ldg(a.b1 + j);
    }
    a.U[(int64_t)c * a.ld1 + j] = acc;
  }
}

__global__ void __launch_bounds__(256) dfm_topn_item_kernel(const DfmTopnArgs a) {
  extern __shared__ float sV[];            // [8][K]
  const int K = a.K;
  const int64_t n0 = (int64_t)blockIdx.x * 8;
  for (int i = threadIdx.x; i < 8 * K; i += blockDim.x) {
    const int64_t n = n0 + i / K;
    sV[i] = (n < a.N) ? __ldg(a.V + (size_t)(a.item_base + n) * K + i % K) : 0.f;
  }
  __syncthreads();
  const float* W = a.W1 + (size_t)a.item_col * K * a.d1;
  for (int j = threadIdx.x; j < a.ld1; j += blockDim.x) {
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (j < a.d1)
      for (int k = 0; k < K; k++) {
        const float w = __ldg(W + (size_t)k * a.d1 + j);
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = fmaf(sV[r * K + k], w, acc[r]);
      }
#pragma unroll
    for (int r = 0; r < 8; r++)
      if (n0 + r < a.N) a.T[(n0 + r) * a.ld1 + j] = acc[r];
  }
}

// X1[c*N + n, :] = relu(U[c] + T[n]) (padding columns stay 0: U and T are 0 there); X1lo (tensor-core path) = its tf32 lo part
__device__ __forceinline__ float dfm_tf32_lo(float x) {      // = tf32_lo of dfm_tc.cu
  const float lo = x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
  return __uint_as_float((__float_as_uint(lo) + 0x1000u) & 0xFFFFE000u);
}

__global__ void __launch_bounds__(256) dfm_topn_h1_kernel(const float* __restrict__ U, const float* __restrict__ T, int64_t C, int64_t N,
                                                          int64_t ld1, float* __restrict__ X1, float* __restrict__ X1lo, int64_t ldx) {
  const int64_t v4 = ld1 >> 2;
  const int64_t total = C * N * v4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = i / v4, j = i % v4;
    const int64_t c = s / N, n = s % N;
    const float4 u = __ldg(reinterpret_cast<const float4*>(U + c * ld1) + j);
    const float4 t = __ldg(reinterpret_cast<const float4*>(T + n * ld1) + j);
    const float4 h = make_float4(fmaxf(u.x + t.x, 0.f), fmaxf(u.y + t.y, 0.f), fmaxf(u.z + t.z, 0.f), fmaxf(u.w + t.w, 0.f));
    reinterpret_cast<float4*>(X1 + s * ldx)[j] = h;
    if (X1lo) reinterpret_cast<float4*>(X1lo + s * ldx)[j] = make_float4(dfm_tf32_lo(h.x), dfm_tf32_lo(h.y), dfm_tf32_lo(h.z), dfm_tf32_lo(h.w));
  }
}

// one warp per (context, item): first order + second order + last hidden layer, through concat_projection (DFM.py:138-143)
// n_part > 0: H holds n_part partial sums of H_L . proj3 per row (TF_EPI_BIAS_RELU_PROJ) instead of H_L itself
__global__ void __launch_bounds__(256) dfm_topn_head_kernel(const DfmTopnArgs a, const float* __restrict__ H, int64_t ldh, int D,
                                                            int n_part, const float* __restrict__ cbias, float* __restrict__ scores) {
  const int lane = threadIdx.x & 31, K = a.K;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t total = (int64_t)a.C * a.N;
  const float cb = __ldg(cbias);
  const float pitem = a.fm ? __ldg(a.proj + a.item_col) : 0.f;
  const float* p2 = a.proj + a.F;
  const float* p3 = a.proj + a.F + K;
  for (int64_t s = warp_g; s < total; s += n_warps) {
    const int64_t c = s / a.N, n = s % a.N;
    const float* v = a.V + (size_t)(a.item_base + n) * K;
    const float* S = a.SQ + c * 2 * K;
    float part = 0.f;
    for (int k = lane; k < (a.fm ? K : 0); k += 32) {
      const float e = __ldg(v + k);
      const float sv = __ldg(S + k) + e, q = fmaf(e, e, __ldg(S + K + k));
      part = fmaf(0.5f * (sv * sv - q), __ldg(p2 + k), part);
    }
    const float* hrow = H + s * ldh;
    if (n_part > 0) {
      if (lane == 0) {
        float d = 0.f;
        for (int q = 0; q < n_part; q++) d += hrow[q];
        part += d;
      }
    } else {
      for (int j = lane; j < D; j += 32) part = fmaf(hrow[j], __ldg(p3 + j), part);
    }
    if (lane == 0 && a.fm) part += __ldg(a.fo + c) + __ldg(a.fbias + a.item_base + n) * pitem;
    const float out = warp_sum(part) + cb;
    if (lane == 0) scores[s] = a.sig ? 1.f / (1.f + expf(-out)) : out;      // what the model's `out` ranks by
  }
}

// side buffers of the evaluator, in this order: U [C, ld1] and T [N, ld1] (tower), SQ [C, 2K] and fo [C] (FM part)
static int64_t dfm_topn_side_floats(int64_t C, int64_t N, int64_t K, int64_t ld1, int32_t mode = 0) {
  return (dfm_deep(mode) ? C * ld1 + N * ld1 : 0) + (dfm_fm(mode) ? C * 2 * K + (C + 3) / 4 * 4 : 0);
}

}  // namespace hhfm

using namespace hhfm;

extern "C" int64_t hhfm_dfm_param_count_mode(int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes, int32_t mode) {
  DfmLayout lo;
  if (dfm_check_mode(mode) != HHFM_OK || dfm_layout(1, F, K, n_layers, layer_sizes, lo, mode) != HHFM_OK) return -1;
  return lo.total;
}

extern "C" int64_t hhfm_dfm_reg_count_mode(int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes, int32_t mode) {
  DfmLayout lo;
  if (dfm_check_mode(mode) != HHFM_OK || dfm_layout(1, F, K, n_layers, layer_sizes, lo, mode) != HHFM_OK) return -1;
  return lo.reg_len;
}

extern "C" int64_t hhfm_dfm_param_count(int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes) {
  return hhfm_dfm_param_count_mode(F, K, n_layers, layer_sizes, 0);
}

extern "C" int64_t hhfm_dfm_reg_count(int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes) {
  return hhfm_dfm_reg_count_mode(F, K, n_layers, layer_sizes, 0);
}

extern "C" int64_t hhfm_workspace_bytes_dfm_mode(int64_t B, int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes,
                                                 int32_t mode) {
  DfmLayout lo;
  if (dfm_check_mode(mode) != HHFM_OK || dfm_layout(B, F, K, n_layers, layer_sizes, lo, mode) != HHFM_OK) return -1;
  if (!dfm_deep(mode)) return 0;               // the head reads nothing but the parameters
  if (dfm_use_tc(K)) {
    DfmTcLayout t;
    dfm_tc_layout(B, lo, t);
    return t.total * (int64_t)sizeof(float);
  }
  return lo.ws_floats * (int64_t)sizeof(float);
}

extern "C" int64_t hhfm_workspace_bytes_dfm(int64_t B, int64_t F, int64_t K, int32_t n_layers,
                                            const int32_t* layer_sizes) {
  return hhfm_workspace_bytes_dfm_mode(B, F, K, n_layers, layer_sizes, 0);
}

// mode: hhfm_dfm_mode bits, or HHFM_DFM_NO_FM | kDfmWd for the Wide&Deep deep part
static int dfm_fwd_impl(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* feature_bias,
                        int64_t M, int64_t K, const float* params, int32_t n_layers, const int32_t* layer_sizes,
                        float* workspace, float* out, hhfm_stream_t stream, int32_t mode, const float* extra) {
  const bool fm = dfm_fm(mode), deep = dfm_deep(mode);
  HHFM_REQUIRE(idx && V && (feature_bias || !fm) && params && (workspace || !deep) && out, "dfm_fwd: NULL argument");
  HHFM_REQUIRE(B >= 0 && B < (1ll << 31) && M > 0, "dfm_fwd: bad sizes");
  if (B == 0) return HHFM_OK;
  DfmLayout lo;
  int rc = dfm_layout(B, F, K, n_layers, layer_sizes, lo, mode);
  if (rc != HHFM_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  HeadArgs h{};
  h.idx = idx; h.B = B; h.F = (int)F; h.K = (int)K; h.D = lo.d[lo.L];
  h.V = V; h.fbias = feature_bias; h.proj = params + lo.proj_off; h.cbias = params + lo.cbias_off; h.out = out;
  dfm_head_mode(mode, h);
  h.extra = extra;
  if (!deep) {                                  // FM part only: no GEMM, no tower input
    h.D = 0; h.H = nullptr; h.ldh = 0;
    return launch_head<false>(h, st);
  }
  if (dfm_use_tc(K)) {
    DfmTcLayout t;
    dfm_tc_layout(B, lo, t);
    HHFM_REQUIRE(((uintptr_t)workspace & 15) == 0, "dfm_fwd: workspace must be 16-byte aligned");
    rc = dfm_tc_forward(idx, B, F, V, K, params, lo, t, workspace, false, st);
    if (rc != HHFM_OK) return rc;
    h.H = workspace + t.x[lo.L]; h.ldh = t.ldx[lo.L];
    return launch_head<false>(h, st);
  }
  rc = dfm_forward(idx, B, F, V, K, params, lo, workspace, st);
  if (rc != HHFM_OK) return rc;
  h.H = workspace + lo.h_off[lo.L]; h.ldh = lo.ld[lo.L];
  return launch_head<false>(h, st);
}

static int dfm_fwd_bwd_impl(const int32_t* idx, int64_t B, int64_t F, const float* V,
                            const float* feature_bias, int64_t M, int64_t K, const float* params,
                            int32_t n_layers, const int32_t* layer_sizes, const float* labels,
                            float* workspace, float* out, float* gV, float* gbias, float* gparams,
                            float* loss_partials, const int32_t* hot_slot, float* ghot, float* ghot_bias,
                            int32_t n_rep, int32_t n_hot, hhfm_stream_t stream, int32_t mode, int64_t B_total,
                            const float* extra, float* gsample) {
  const bool fm = dfm_fm(mode), deep = dfm_deep(mode);
  HHFM_REQUIRE(idx && V && (feature_bias || !fm) && params && (workspace || !deep) && labels && gV && (gbias || !fm) && gparams &&
               loss_partials, "dfm_fwd_bwd: NULL argument");
  HHFM_REQUIRE(B > 0 && B < (1ll << 31) && M > 0, "dfm_fwd_bwd: bad sizes");
  HHFM_REQUIRE(B_total >= B, "dfm_fwd_bwd: B_total (%lld) must be >= B (%lld)", (long long)B_total, (long long)B);
  DfmLayout lo;
  int rc = dfm_layout(B, F, K, n_layers, layer_sizes, lo, mode);
  if (rc != HHFM_OK) return rc;
  HHFM_REQUIRE(!hot_slot || (ghot && n_rep >= 1 && n_hot >= 1), "dfm_fwd_bwd: hot_slot needs ghot, n_rep, n_hot");
  cudaStream_t st = (cudaStream_t)stream;
  const int L = lo.L;
  const HotPlan hot{hot_slot, ghot, ghot_bias, n_rep, n_hot};
  HeadArgs h{};
  h.idx = idx; h.B = B; h.F = (int)F; h.K = (int)K; h.D = lo.d[L];
  h.V = V; h.fbias = feature_bias; h.proj = params + lo.proj_off; h.cbias = params + lo.cbias_off;
  h.labels = labels; h.out = out;
  h.gV = gV; h.gfbias = gbias; h.gproj = gparams + lo.proj_off; h.gcbias = gparams + lo.cbias_off;
  h.gblast = gparams + lo.b_off[L - 1]; h.loss_partials = loss_partials; h.hot = hot;
  dfm_head_mode(mode, h);
  h.extra = extra; h.gsample = gsample; h.inv_b = 1.0f / (float)B_total;
  if (!deep) {                                  // FM part only: D = 0, no dZ, no tower gradients
    h.D = 0; h.H = nullptr; h.ldh = 0; h.gblast = nullptr;
    return launch_head<true>(h, st);
  }
  if (dfm_use_tc(K)) {
    DfmTcLayout t;
    dfm_tc_layout(B, lo, t);
    HHFM_REQUIRE(((uintptr_t)workspace & 15) == 0, "dfm_fwd_bwd: workspace must be 16-byte aligned");
    float* ws = workspace;
    if ((rc = dfm_tc_forward(idx, B, F, V, K, params, lo, t, ws, true, st))) return rc;
    h.H = ws + t.x[L]; h.ldh = t.ldx[L];
    if ((rc = launch_head<true>(h, st))) return rc;
    // dZ_L (in the X_L block) -> lo / transposed forms
    if ((rc = tf_split_transpose(ws + t.x[L], B, lo.d[L], t.ldx[L], ws + t.xlo[L], ws + t.xt[L], ws + t.xtlo[L], st))) return rc;
    for (int i = L - 1; i >= 0; i--) {
      // bias gradient of layer i (the head kernel already produced the last one)
      if (i < L - 1 && (rc = tf_colsum(ws + t.x[i + 1], B, lo.d[i + 1], t.ldx[i + 1], gparams + lo.b_off[i], st))) return rc;
      // d layer_i = H_i^T . dZ_{i+1}: A = X_i^T [d_i, B], B = dZ_{i+1}^T [d_{i+1}, B], split over the samples
      TfGemm w{};
      w.A = ws + t.xt[i]; w.A_lo = ws + t.xtlo[i]; w.B = ws + t.xt[i + 1]; w.B_lo = ws + t.xtlo[i + 1]; w.k_blocked = 1;
      w.M = lo.d[i]; w.N = lo.d[i + 1]; w.K = (int)B;
      w.epi = TF_EPI_ATOMIC; w.C = gparams + lo.w_off[i]; w.ldc = lo.d[i + 1];
      w.scratch = ws + t.scratch; w.scratch_floats = t.scratch_floats;
      if ((rc = tf_gemm(w, st))) return rc;
      // d H_i = dZ_{i+1} . layer_i^T: A = dZ_{i+1} [B, d_{i+1}], B = layer_i [d_i, d_{i+1}]
      TfGemm x{};
      x.A = ws + t.x[i + 1]; x.A_lo = ws + t.xlo[i + 1]; x.lda = t.ldx[i + 1];
      x.B = ws + t.w[i]; x.B_lo = ws + t.wlo[i]; x.ldb = t.ldp[i];
      x.M = (int)B; x.N = lo.d[i]; x.K = lo.d[i + 1];
      if (i == 0) {
        x.epi = TF_EPI_SCATTER; x.C = gV; x.idx = idx; x.F = (int)F; x.Kemb = (int)K; x.hot = hot;
        if ((rc = tf_gemm(x, st))) return rc;
      } else {
        // unmasked product into the (no longer needed) lo block of H_i; the split pass applies relu'(H_i) and leaves dZ_i in
        // the H_i block, its lo part in the lo block and the k-blocked transposes
        x.epi = TF_EPI_STORE; x.C = ws + t.xlo[i]; x.ldc = t.ldx[i];
        if ((rc = tf_gemm(x, st))) return rc;
        if ((rc = tf_split_transpose(ws + t.xlo[i], B, lo.d[i], t.ldx[i], ws + t.xlo[i], ws + t.xt[i], ws + t.xtlo[i], st,
                                     ws + t.x[i], ws + t.x[i])))
          return rc;
      }
    }
    return HHFM_OK;
  }
  rc = dfm_forward(idx, B, F, V, K, params, lo, workspace, st);
  if (rc != HHFM_OK) return rc;
  h.H = workspace + lo.h_off[L]; h.ldh = lo.ld[L];
  rc = launch_head<true>(h, st);
  if (rc != HHFM_OK) return rc;
  // backward through the tower: layer i maps H_i -> H_{i+1}; dZ_{i+1} lives in the H_{i+1} block
  for (int i = L - 1; i >= 0; i--) {
    const float* dZ = workspace + lo.h_off[i + 1];
    // d layer_i = H_i^T dZ_{i+1}   (split-K over the samples)
    GemmArgs w{};
    w.M = lo.d[i]; w.N = lo.d[i + 1]; w.Kd = (int)B;
    w.B = dZ; w.ldb = lo.ld[i + 1];
    w.C = gparams + lo.w_off[i]; w.ldc = lo.d[i + 1];
    if (i == 0) {
      w.A = V; w.idx = idx; w.F = (int)F; w.K = (int)K;
      rc = launch_gemm<A_GATHER_T, B_ROW, EPI_ATOMIC>(w, st);
    } else {
      w.A = workspace + lo.h_off[i]; w.lda = lo.ld[i];
      rc = launch_gemm<A_COL, B_ROW, EPI_ATOMIC>(w, st);
    }
    if (rc != HHFM_OK) return rc;
    // d H_i = dZ_{i+1} layer_i^T, masked by relu'(H_i) (in place), or scattered into the embedding gradient (i == 0)
    GemmArgs x{};
    x.M = (int)B; x.N = lo.d[i]; x.Kd = lo.d[i + 1];
    x.A = dZ; x.lda = lo.ld[i + 1];
    x.B = params + lo.w_off[i]; x.ldb = lo.d[i + 1];
    if (i == 0) {
      x.C = gV; x.idx = idx; x.F = (int)F; x.K = (int)K; x.hot = hot;
      rc = launch_gemm<A_ROW, B_COL, EPI_SCATTER>(x, st);
    } else {
      x.C = workspace + lo.h_off[i]; x.ldc = lo.ld[i];
      x.mask = x.C; x.ldmask = lo.ld[i];
      x.colsum = gparams + lo.b_off[i - 1];
      rc = launch_gemm<A_ROW, B_COL, EPI_MASK>(x, st);
    }
    if (rc != HHFM_OK) return rc;
  }
  return HHFM_OK;
}

extern "C" int hhfm_dfm_fwd_mode(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* feature_bias, int64_t M,
                                 int64_t K, const float* params, int32_t n_layers, const int32_t* layer_sizes, int32_t mode,
                                 float* workspace, float* out, hhfm_stream_t stream) {
  int rc = dfm_check_mode(mode);
  if (rc != HHFM_OK) return rc;
  return dfm_fwd_impl(idx, B, F, V, feature_bias, M, K, params, n_layers, layer_sizes, workspace, out, stream, mode, nullptr);
}

extern "C" int hhfm_dfm_fwd_bwd_mode(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* feature_bias,
                                     int64_t M, int64_t K, const float* params, int32_t n_layers, const int32_t* layer_sizes,
                                     int32_t mode, int64_t B_total, const float* labels, float* workspace, float* out, float* gV,
                                     float* gbias, float* gparams, float* loss_partials, const int32_t* hot_slot, float* ghot,
                                     float* ghot_bias, int32_t n_rep, int32_t n_hot, hhfm_stream_t stream) {
  int rc = dfm_check_mode(mode);
  if (rc != HHFM_OK) return rc;
  return dfm_fwd_bwd_impl(idx, B, F, V, feature_bias, M, K, params, n_layers, layer_sizes, labels, workspace, out, gV, gbias,
                          gparams, loss_partials, hot_slot, ghot, ghot_bias, n_rep, n_hot, stream, mode, B_total, nullptr, nullptr);
}

extern "C" int hhfm_dfm_fwd(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* feature_bias,
                            int64_t M, int64_t K, const float* params, int32_t n_layers, const int32_t* layer_sizes,
                            float* workspace, float* out, hhfm_stream_t stream) {
  return hhfm_dfm_fwd_mode(idx, B, F, V, feature_bias, M, K, params, n_layers, layer_sizes, 0, workspace, out, stream);
}

extern "C" int hhfm_dfm_fwd_bwd_sqloss(const int32_t* idx, int64_t B, int64_t F, const float* V,
                                       const float* feature_bias, int64_t M, int64_t K, const float* params,
                                       int32_t n_layers, const int32_t* layer_sizes, const float* labels,
                                       float* workspace, float* out, float* gV, float* gbias, float* gparams,
                                       float* loss_partials, const int32_t* hot_slot, float* ghot, float* ghot_bias,
                                       int32_t n_rep, int32_t n_hot, hhfm_stream_t stream) {
  return hhfm_dfm_fwd_bwd_mode(idx, B, F, V, feature_bias, M, K, params, n_layers, layer_sizes, 0, B, labels, workspace, out, gV,
                               gbias, gparams, loss_partials, hot_slot, ghot, ghot_bias, n_rep, n_hot, stream);
}

// Wide&Deep deep part (WDMF.py:57-73): the DeepFM tower with its FM terms off; `extra` [B] is the wide logit, `out` the summed
// logit, `gsample` [B] receives d(mean log-loss)/d logit for the wide part's backward.  Parameter block: the DeepFM layout
// (the first F + K entries of the projection block are unused and stay zero).
extern "C" int hhfm_wd_deep_fwd(const int32_t* idx, int64_t B, int64_t F, const float* V, int64_t M, int64_t K,
                                const float* params, int32_t n_layers, const int32_t* layer_sizes, const float* extra,
                                float* workspace, float* out, hhfm_stream_t stream) {
  return dfm_fwd_impl(idx, B, F, V, nullptr, M, K, params, n_layers, layer_sizes, workspace, out, stream, HHFM_DFM_NO_FM | kDfmWd,
                      extra);
}

extern "C" int hhfm_wd_deep_fwd_bwd_logloss(const int32_t* idx, int64_t B, int64_t F, const float* V, int64_t M, int64_t K,
                                            const float* params, int32_t n_layers, const int32_t* layer_sizes,
                                            const float* labels, const float* extra, float* workspace, float* out,
                                            float* gV, float* gparams, float* gsample, float* loss_partials,
                                            const int32_t* hot_slot, float* ghot, int32_t n_rep, int32_t n_hot,
                                            hhfm_stream_t stream) {
  return dfm_fwd_bwd_impl(idx, B, F, V, nullptr, M, K, params, n_layers, layer_sizes, labels, workspace, out, gV, nullptr, gparams,
                          loss_partials, hot_slot, ghot, nullptr, n_rep, n_hot, stream, HHFM_DFM_NO_FM | kDfmWd, B, extra, gsample);
}

extern "C" int64_t hhfm_workspace_bytes_dfm_topn_mode(int64_t C, int64_t N, int64_t F, int64_t K, int32_t n_layers,
                                                      const int32_t* layer_sizes, int32_t mode) {
  DfmLayout lo;
  if (dfm_check_mode(mode) != HHFM_OK) return -1;
  if (C < 0 || N < 1 || dfm_layout(C * N, F, K, n_layers, layer_sizes, lo, mode) != HHFM_OK) return -1;
  const int64_t side = dfm_topn_side_floats(C, N, K, lo.ld[1], mode);
  if (!dfm_deep(mode)) return side * (int64_t)sizeof(float);      // no tower activations for the C*N rows
  if (dfm_use_tc(K)) {
    DfmTcLayout t;
    dfm_tc_layout(C * N, lo, t, 1);
    return (side + t.total) * (int64_t)sizeof(float);
  }
  return (side + lo.ws_floats) * (int64_t)sizeof(float);
}

extern "C" int64_t hhfm_workspace_bytes_dfm_topn(int64_t C, int64_t N, int64_t F, int64_t K, int32_t n_layers,
                                                 const int32_t* layer_sizes) {
  return hhfm_workspace_bytes_dfm_topn_mode(C, N, F, K, n_layers, layer_sizes, 0);
}

extern "C" int hhfm_dfm_topn_scores_mode(const int32_t* rows, int64_t row_stride, int64_t C, int64_t F, int32_t item_col,
                                         const float* V, const float* feature_bias, int64_t M, int64_t K, const float* params,
                                         int32_t n_layers, const int32_t* layer_sizes, int32_t mode, int64_t item_base, int64_t N,
                                         float* workspace, float* scores, hhfm_stream_t stream) {
  int rc = dfm_check_mode(mode);
  if (rc != HHFM_OK) return rc;
  const bool fm = dfm_fm(mode), deep = dfm_deep(mode);
  HHFM_REQUIRE(rows && V && (feature_bias || !fm) && params && workspace && scores, "dfm_topn_scores: NULL argument");
  HHFM_REQUIRE(C >= 0 && N >= 1 && C * N < (1ll << 31) && item_base >= 0 && item_base + N <= M, "dfm_topn_scores: bad C / N / item_base");
  HHFM_REQUIRE(item_col >= 0 && item_col < F && row_stride >= F, "dfm_topn_scores: bad item_col / row_stride");
  HHFM_REQUIRE(((uintptr_t)workspace & 15) == 0, "dfm_topn_scores: workspace must be 16-byte aligned");
  if (C == 0) return HHFM_OK;
  const int64_t B = C * N;
  DfmLayout lo;
  rc = dfm_layout(B, F, K, n_layers, layer_sizes, lo, mode);
  if (rc != HHFM_OK) return rc;
  HHFM_REQUIRE(F * K * sizeof(float) <= 200 * 1024, "dfm_topn_scores: F*K too large for the context kernel");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t ld1 = lo.ld[1];
  DfmTopnArgs a{};
  a.rows = rows; a.row_stride = row_stride; a.C = (int)C; a.F = (int)F; a.K = (int)K; a.item_col = item_col; a.d1 = lo.d[1]; a.ld1 = ld1;
  a.V = V; a.fbias = feature_bias; a.W1 = params + lo.w_off[0]; a.b1 = params + lo.b_off[0]; a.proj = params + lo.proj_off;
  a.item_base = item_base; a.N = N;
  a.fm = fm ? 1 : 0; a.deep = deep ? 1 : 0; a.sig = (mode & HHFM_DFM_LOGLOSS) ? 1 : 0;
  a.U = workspace; a.T = a.U + (deep ? C * ld1 : 0); a.SQ = a.T + (deep ? N * ld1 : 0); a.fo = a.SQ + C * 2 * K;
  float* main_ws = workspace + dfm_topn_side_floats(C, N, K, ld1, mode);
  {
    const size_t smem = (size_t)F * K * sizeof(float);
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(dfm_topn_ctx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      set_error("dfm_topn_ctx_kernel: cannot reserve %zu bytes of shared memory", smem);
      return HHFM_ERR_LAUNCH;
    }
    dfm_topn_ctx_kernel<<<(unsigned)C, 256, smem, st>>>(a);
    if ((rc = check_launch("dfm_topn_ctx_kernel"))) return rc;
    if (deep) {
      dfm_topn_item_kernel<<<(unsigned)((N + 7) / 8), 256, 8 * K * sizeof(float), st>>>(a);
      if ((rc = check_launch("dfm_topn_item_kernel"))) return rc;
    }
  }
  const float* H = nullptr;
  int64_t ldh = 0;
  int n_part = 0, D = 0;
  const int h1_grid = (int)std::min<int64_t>((B * (ld1 >> 2) + 255) / 256, (int64_t)sm_count() * 16);
  // FM part only (!deep): the head kernel reads SQ / fo and the item's row; nothing per (row, item) is materialised
  if (deep && dfm_use_tc(K)) {
    DfmTcLayout t;
    dfm_tc_layout(B, lo, t, 1);
    dfm_topn_h1_kernel<<<h1_grid, 256, 0, st>>>(a.U, a.T, C, N, ld1, main_ws + t.x[1], main_ws + t.xlo[1], t.ldx[1]);
    if ((rc = check_launch("dfm_topn_h1_kernel"))) return rc;
    const bool fuse_proj = lo.L >= 2 && tf_proj_partials(lo.d[lo.L]) <= t.ldx[lo.L];
    if ((rc = dfm_tc_forward(nullptr, B, F, V, K, params, lo, t, main_ws, false, st, 1, true,
                             fuse_proj ? params + lo.proj_off + F + K : nullptr)))
      return rc;
    H = main_ws + t.x[lo.L]; ldh = t.ldx[lo.L]; D = lo.d[lo.L];
    n_part = fuse_proj ? tf_proj_partials(lo.d[lo.L]) : 0;
  } else if (deep) {
    dfm_topn_h1_kernel<<<h1_grid, 256, 0, st>>>(a.U, a.T, C, N, ld1, main_ws + lo.h_off[1], nullptr, lo.ld[1]);
    if ((rc = check_launch("dfm_topn_h1_kernel"))) return rc;
    if ((rc = dfm_forward(nullptr, B, F, V, K, params, lo, main_ws, st, 1))) return rc;
    H = main_ws + lo.h_off[lo.L]; ldh = lo.ld[lo.L]; D = lo.d[lo.L];
  }
  const int head_grid = (int)std::min<int64_t>((B + 7) / 8, (int64_t)sm_count() * 8);
  dfm_topn_head_kernel<<<head_grid, 256, 0, st>>>(a, H, ldh, D, n_part, params + lo.cbias_off, scores);
  return check_launch("dfm_topn_head_kernel");
}

extern "C" int hhfm_dfm_topn_scores(const int32_t* rows, int64_t row_stride, int64_t C, int64_t F, int32_t item_col,
                                    const float* V, const float* feature_bias, int64_t M, int64_t K, const float* params,
                                    int32_t n_layers, const int32_t* layer_sizes, int64_t item_base, int64_t N,
                                    float* workspace, float* scores, hhfm_stream_t stream) {
  return hhfm_dfm_topn_scores_mode(rows, row_stride, C, F, item_col, V, feature_bias, M, K, params, n_layers, layer_sizes, 0,
                                   item_base, N, workspace, scores, stream);
}
