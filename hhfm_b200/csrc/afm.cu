// K2: Attentional FM (Newcode/AFM.py:103-148), fp32 SIMT, forward and fused forward + squared loss + backward.
//
//   E = V[x] [F,K];  P_p = E_i * E_j for the pairs i<j in lexicographic order (AFM.py:105-112), never materialised in HBM
//   Z_p = P_p W + b (W [K,A]);  s_p = relu(Z_p) . p;  a = softmax_p(s)  (AFM.py:117-125)
//   afm = sum_p a_p P_p;  out = afm . w_pred + sum_f bias[x_f] + b0      (AFM.py:130-142)
//   loss = 0.5 sum (y - out)^2  (+ lamda_attention/2 ||W||^2 is added by the caller through the dense-L2 optimizer)
//
// One warp owns one sample; a CTA of NW warps works on NW samples at a time.  W lives in shared memory with a padded
// row (A+1) so that both the forward (lanes over a) and the backward (lanes over k) read it without bank conflicts.
// The weight gradient dW = sum P_p^T dZ_p is accumulated in REGISTERS: warp w owns the k-slice [w K/NW, (w+1) K/NW)
// and, after a CTA barrier, sweeps the (E, dZ) of all NW samples of the tile from shared memory.  Embedding gradients
// go through the same sort-free vector reductions (and hot-row replicas) as the FM / HHFM kernels.
// These kernels are compute-bound (about 1.1 MFLOP per sample at F=10, K=A=64) and serve every shape; the training pass of the
// reference's default shape family (K = A = 64, F <= 11) runs on the tensor cores instead (afm_fused_tc.cu).
#include <stdlib.h>

#include "afm.cuh"
#include "common.cuh"

namespace hhfm {

// drop: the DROP instantiations keep the sample's attention-dropout factors m_p in one more row of P floats
__host__ __device__ inline size_t afm_per_warp_floats(int F, int K, int A, int P, bool drop = false) {
  return 2 * (size_t)F * K + (size_t)P * A + (size_t)((2 * P + 3) / 4 * 4) + (drop ? (size_t)((P + 3) / 4 * 4) : 0);
}

__host__ __device__ inline size_t afm_smem_floats(int NW, int F, int K, int A, int P, bool drop = false) {
  // sW[K][A+1] + sp[A] + sb[A] + swp[K] + NW * (sE[F][K] + sDE[F][K] + sZ[P][A] + sS[P] + sD[P] (padded) [+ sM[P]]) + valid flags
  return (size_t)K * (A + 1) + 2 * (size_t)A + K + (size_t)NW * afm_per_warp_floats(F, K, A, P, drop) + 32;
}

constexpr int PB = 8;       // pairs per register-blocked sweep of the two matrix products

// DROP: training dropout (AFM.py:126,134).  a_p m_p replaces a_p in the pooled sum, w~ = prediction_W * n replaces
// prediction_W, d prediction_W += g n afm, and the softmax backward becomes ds_p = a_p (m_p d a_p - sum_q a_q m_q d a_q).
template <int TK, int TA, int NW, bool TRAIN, bool DROP = false>
__global__ void __launch_bounds__(NW * 32) afm_kernel(const AfmArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float scratch[32];
  const int K = a.K, A = a.A, F = a.F, P = a.P;
  const int AS = A + 1;
  float* sW = smem;                       // [K][A+1]
  float* sp = sW + (size_t)K * AS;        // [A]
  float* sb = sp + A;                     // [A]
  float* swp = sb + A;                    // [K]
  float* warp_base = swp + K;
  const size_t per_warp = afm_per_warp_floats(F, K, A, P, DROP);
  int* sValid = reinterpret_cast<int*>(warp_base + (size_t)NW * per_warp);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sE = warp_base + warp * per_warp;   // [F][K]
  float* sDE = sE + (size_t)F * K;           // [F][K]  d E accumulated over the pairs
  float* sZ = sDE + (size_t)F * K;           // [P][A]  Z, later dZ
  float* sS = sZ + (size_t)P * A;            // [P]     s, later a
  float* sD = sS + P;                        // [P]     d a, later d s
  float* sM = sS + (2 * P + 3) / 4 * 4;      // [P]     m_p (DROP)
  const uint64_t vseed = DROP ? splitmix64(a.drop_seed) : 0;

  for (int i = threadIdx.x; i < K * A; i += blockDim.x) sW[(i / A) * AS + (i % A)] = __ldg(a.W + i);
  for (int i = threadIdx.x; i < A; i += blockDim.x) { sp[i] = __ldg(a.pvec + i); sb[i] = __ldg(a.batt + i); }
  for (int i = threadIdx.x; i < K; i += blockDim.x) swp[i] = __ldg(a.wpred + i);
  __syncthreads();

  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  const int rep = a.hot.slot ? (int)(((int64_t)blockIdx.x * NW + warp) % a.hot.n_rep) : 0;
  // pair table (i,j) packed as i*16+j, computed once per warp into registers-of-smem: reuse scratch-free small array
  __shared__ unsigned char sPairI[kAfmMaxP], sPairJ[kAfmMaxP];
  if (threadIdx.x == 0) {
    int p = 0;
    for (int i = 0; i < F; i++)
      for (int j = i + 1; j < F; j++) { sPairI[p] = (unsigned char)i; sPairJ[p] = (unsigned char)j; p++; }
  }
  __syncthreads();

  // persistent accumulators
  constexpr int KSMAX = (32 * TK) / NW;              // k-slice rows per warp (K <= 32*TK)
  float dWacc[TRAIN ? KSMAX : 1][TA];
  float gbatt_acc[TA], gp_acc[TA], gwp_acc[TK];
  float loss_acc = 0.f, g0_acc = 0.f;
  if (TRAIN) {
#pragma unroll
    for (int r = 0; r < KSMAX; r++)
#pragma unroll
      for (int t = 0; t < TA; t++) dWacc[r][t] = 0.f;
  }
#pragma unroll
  for (int t = 0; t < TA; t++) { gbatt_acc[t] = 0.f; gp_acc[t] = 0.f; }
#pragma unroll
  for (int t = 0; t < TK; t++) gwp_acc[t] = 0.f;
  const int KS = K / NW;                             // host guarantees K % NW == 0

  for (int64_t s0 = (int64_t)blockIdx.x * NW; s0 < a.B; s0 += (int64_t)gridDim.x * NW) {
    const int64_t s = s0 + warp;
    const bool valid = s < a.B;
    if (lane == 0) sValid[warp] = valid ? 1 : 0;
    if (valid) {
      const int32_t* rec = a.idx + s * F;
      // ---- gather E (coalesced float4 rows) and the bias sum ----
      float bsum = 0.f;
      for (int f = 0; f < F; f++) {
        const int id = __ldg(rec + f);
        const float4* src = reinterpret_cast<const float4*>(a.V + (size_t)id * K);
        for (int c = lane; c < (K >> 2); c += 32) reinterpret_cast<float4*>(sE + f * K)[c] = __ldg(src + c);
        if (a.bias) bsum += __ldg(a.bias + id);
      }
      __syncwarp();
      // ---- attention logits: Z_p = P_p W + b, s_p = relu(Z_p) . p   (4 pairs per sweep over k) ----
      for (int p0 = 0; p0 < P; p0 += PB) {
        float acc[PB][TA];
#pragma unroll
        for (int q = 0; q < PB; q++)
#pragma unroll
          for (int t = 0; t < TA; t++) acc[q][t] = (lane + 32 * t < A) ? sb[lane + 32 * t] : 0.f;
        const float* ei[PB]; const float* ej[PB];
#pragma unroll
        for (int q = 0; q < PB; q++) {
          const int p = min(p0 + q, P - 1);
          ei[q] = sE + sPairI[p] * K; ej[q] = sE + sPairJ[p] * K;
        }
        for (int k = 0; k < K; k += 4) {
          float pk[PB][4];
#pragma unroll
          for (int q = 0; q < PB; q++) {
            const float4 x = *reinterpret_cast<const float4*>(ei[q] + k);
            const float4 y = *reinterpret_cast<const float4*>(ej[q] + k);
            pk[q][0] = x.x * y.x; pk[q][1] = x.y * y.y; pk[q][2] = x.z * y.z; pk[q][3] = x.w * y.w;
          }
#pragma unroll
          for (int kk = 0; kk < 4; kk++) {
#pragma unroll
            for (int t = 0; t < TA; t++) {
              const int aa = lane + 32 * t;
              const float w = (aa < A) ? sW[(k + kk) * AS + aa] : 0.f;
#pragma unroll
              for (int q = 0; q < PB; q++) acc[q][t] = fmaf(pk[q][kk], w, acc[q][t]);
            }
          }
        }
#pragma unroll
        for (int q = 0; q < PB; q++) {
          const int p = p0 + q;
          if (p < P) {
            float part = 0.f;
#pragma unroll
            for (int t = 0; t < TA; t++) {
              const int aa = lane + 32 * t;
              if (aa < A) {
                sZ[p * A + aa] = acc[q][t];
                part = fmaf(fmaxf(acc[q][t], 0.f), sp[aa], part);
              }
            }
            part = warp_sum(part);
            if (lane == 0) sS[p] = part;
          }
        }
      }
      __syncwarp();
      // ---- softmax over pairs (AFM.py:125) ----
      float mx = -INFINITY;
      for (int p = lane; p < P; p += 32) mx = fmaxf(mx, sS[p]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float den = 0.f;
      for (int p = lane; p < P; p += 32) { const float e = expf(sS[p] - mx); sS[p] = e; den += e; }
      den = warp_sum(den);
      __syncwarp();
      for (int p = lane; p < P; p += 32) {
        sS[p] = sS[p] / den;
        if (DROP) sM[p] = afm_mask_att(a, s, p) / a.keep_att;
      }
      __syncwarp();
      float nv[TK];                                               // n_k of the lane's columns (DROP)
#pragma unroll
      for (int t = 0; t < TK; t++) nv[t] = DROP ? afm_mask_vec(a, vseed, s, lane + 32 * t) / a.keep_vec : 1.f;
      // ---- afm = sum_p a_p P_p (lanes over k), out ----
      float afm[TK];
#pragma unroll
      for (int t = 0; t < TK; t++) afm[t] = 0.f;
      for (int p = 0; p < P; p++) {
        const float ap = DROP ? sS[p] * sM[p] : sS[p];
        const float* xi = sE + sPairI[p] * K; const float* xj = sE + sPairJ[p] * K;
#pragma unroll
        for (int t = 0; t < TK; t++) {
          const int k = lane + 32 * t;
          if (k < K) afm[t] = fmaf(ap, xi[k] * xj[k], afm[t]);
        }
      }
      float part = 0.f;
#pragma unroll
      for (int t = 0; t < TK; t++) { const int k = lane + 32 * t; if (k < K) part = fmaf(afm[t], DROP ? swp[k] * nv[t] : swp[k], part); }
      const float bil = warp_sum(part);
      const float out = (bil + bsum) + b0;                       // AFM.py:142 add_n
      if (a.out && lane == 0) a.out[s] = out;

      if (TRAIN) {
        const float y = __ldg(a.labels + s);
        const float diff = y - out;
        const float g = -diff;
        if (lane == 0) { loss_acc += 0.5f * diff * diff; g0_acc += g; }
        // d afm = g w_pred ; d w_pred += g afm   (DROP: w~ = w_pred n, d w_pred += g n afm)
        float dafm[TK];
#pragma unroll
        for (int t = 0; t < TK; t++) {
          const int k = lane + 32 * t;
          dafm[t] = (k < K) ? g * (DROP ? swp[k] * nv[t] : swp[k]) : 0.f;
          gwp_acc[t] = fmaf(g, DROP ? afm[t] * nv[t] : afm[t], gwp_acc[t]);
        }
        // d a_p = P_p . d afm ; softmax backward
        float dot = 0.f;
        for (int p = 0; p < P; p++) {
          const float* xi = sE + sPairI[p] * K; const float* xj = sE + sPairJ[p] * K;
          float v = 0.f;
#pragma unroll
          for (int t = 0; t < TK; t++) { const int k = lane + 32 * t; if (k < K) v = fmaf(xi[k] * xj[k], dafm[t], v); }
          v = warp_sum(v);
          if (lane == 0) sD[p] = v;
          dot = fmaf(DROP ? sS[p] * sM[p] : sS[p], v, dot);
        }
        __syncwarp();
        for (int p = lane; p < P; p += 32) sD[p] = sS[p] * ((DROP ? sM[p] * sD[p] : sD[p]) - dot);       // d s_p
        __syncwarp();
        // d Z_p = d s_p p (Z_p > 0) (overwrites Z) ; d p += d s_p relu(Z_p) ; d b += d Z_p
        for (int p = 0; p < P; p++) {
          const float ds = sD[p];
#pragma unroll
          for (int t = 0; t < TA; t++) {
            const int aa = lane + 32 * t;
            if (aa < A) {
              const float z = sZ[p * A + aa];
              const float dz = (z > 0.f) ? ds * sp[aa] : 0.f;
              gp_acc[t] = fmaf(ds, fmaxf(z, 0.f), gp_acc[t]);
              gbatt_acc[t] += dz;
              sZ[p * A + aa] = dz;
            }
          }
        }
        __syncwarp();
        // d P_p = a_p d afm + W d Z_p (lanes over k, 4 pairs per sweep over a) ; d E_i += dP*E_j ; d E_j += dP*E_i
        for (int i = lane; i < F * K; i += 32) sDE[i] = 0.f;
        __syncwarp();
        for (int p0 = 0; p0 < P; p0 += PB) {
          float dp[PB][TK];
#pragma unroll
          for (int q = 0; q < PB; q++) {
            const float ap = (p0 + q < P) ? (DROP ? sS[p0 + q] * sM[p0 + q] : sS[p0 + q]) : 0.f;
#pragma unroll
            for (int t = 0; t < TK; t++) dp[q][t] = ap * dafm[t];
          }
          for (int a0 = 0; a0 < A; a0 += 4) {
            float dz[PB][4];
#pragma unroll
            for (int q = 0; q < PB; q++) {
              const float4 v = *reinterpret_cast<const float4*>(sZ + min(p0 + q, P - 1) * A + a0);
              dz[q][0] = v.x; dz[q][1] = v.y; dz[q][2] = v.z; dz[q][3] = v.w;
            }
#pragma unroll
            for (int aa = 0; aa < 4; aa++) {
#pragma unroll
              for (int t = 0; t < TK; t++) {
                const int k = lane + 32 * t;
                const float w = (k < K) ? sW[k * AS + a0 + aa] : 0.f;
#pragma unroll
                for (int q = 0; q < PB; q++) dp[q][t] = fmaf(w, dz[q][aa], dp[q][t]);
              }
            }
          }
#pragma unroll
          for (int q = 0; q < PB; q++) {
            const int p = p0 + q;
            if (p < P) {
              const int fi = sPairI[p], fj = sPairJ[p];
#pragma unroll
              for (int t = 0; t < TK; t++) {
                const int k = lane + 32 * t;
                if (k < K) {                 // the warp is the only writer of sDE and lane k owns column k
                  const float xi = sE[fi * K + k], xj = sE[fj * K + k];
                  sDE[fi * K + k] = fmaf(dp[q][t], xj, sDE[fi * K + k]);
                  sDE[fj * K + k] = fmaf(dp[q][t], xi, sDE[fj * K + k]);
                }
              }
            }
          }
        }
        // scatter d E rows (vector reductions), d bias
        __syncwarp();
        for (int f = 0; f < F; f++) {
          const int id = __ldg(rec + f);
          float* dst = a.gV + (size_t)id * K;
          if (a.hot.slot != nullptr) {
            const int hs = __ldg(a.hot.slot + id);
            if (hs >= 0) dst = a.hot.ghot + ((size_t)rep * a.hot.n_hot + hs) * K;
          }
          for (int c = lane; c < (K >> 2); c += 32) red_add_v4(dst + 4 * c, reinterpret_cast<const float4*>(sDE + f * K)[c]);
          if (lane == 0) {
            if (a.gbias) scatter_bias(a.gbias, a.hot, rep, id, g);
            touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, id);
          }
        }
      }
    }
    if (TRAIN) {
      __syncthreads();
      // ---- d W: warp w owns k in [w*KS, (w+1)*KS); sweep (E, dZ) of every valid sample of this tile ----
      for (int ws = 0; ws < NW; ws++) {
        if (!sValid[ws]) continue;
        const float* oE = warp_base + ws * per_warp;
        const float* oZ = oE + 2 * (size_t)F * K;
        for (int p = 0; p < P; p++) {
          float dz[TA];
#pragma unroll
          for (int t = 0; t < TA; t++) { const int aa = lane + 32 * t; dz[t] = (aa < A) ? oZ[p * A + aa] : 0.f; }
          const float* xi = oE + sPairI[p] * K + warp * KS; const float* xj = oE + sPairJ[p] * K + warp * KS;
#pragma unroll
          for (int r = 0; r < KSMAX; r += 4) {
            if (r < KS) {
              const float4 x = *reinterpret_cast<const float4*>(xi + r);
              const float4 y = *reinterpret_cast<const float4*>(xj + r);
              const float pk[4] = {x.x * y.x, x.y * y.y, x.z * y.z, x.w * y.w};
#pragma unroll
              for (int rr = 0; rr < 4; rr++)
#pragma unroll
                for (int t = 0; t < TA; t++) dWacc[r + rr][t] = fmaf(pk[rr], dz[t], dWacc[r + rr][t]);
            }
          }
        }
      }
      __syncthreads();
    }
  }

  if (TRAIN) {
    // flush the register accumulators
#pragma unroll
    for (int r = 0; r < KSMAX; r++) {
      if (r < KS) {
#pragma unroll
        for (int t = 0; t < TA; t++) {
          const int aa = lane + 32 * t;
          if (aa < A && dWacc[r][t] != 0.f) atomicAdd(a.gW + (size_t)(warp * KS + r) * A + aa, dWacc[r][t]);
        }
      }
    }
#pragma unroll
    for (int t = 0; t < TA; t++) {
      const int aa = lane + 32 * t;
      if (aa < A) { atomicAdd(a.gbatt + aa, gbatt_acc[t]); atomicAdd(a.gp + aa, gp_acc[t]); }
    }
#pragma unroll
    for (int t = 0; t < TK; t++) { const int k = lane + 32 * t; if (k < K) atomicAdd(a.gwpred + k, gwp_acc[t]); }
    const float bl = block_sum(loss_acc, scratch);
    write_partial(a.loss_partials, bl);
    const float bg = block_sum(g0_acc, scratch);
    if (threadIdx.x == 0 && a.gb0 && bg != 0.f) atomicAdd(a.gb0, bg);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Second layout (K == A == KD in {16, 32, 64}): ONE LANE PER PAIR for the two row-times-matrix products.
// In afm_kernel the lanes run over the attention columns, so every FMA group needs its own W loads (ncu: 3.3 instructions
// per FMA, FMA pipe 29 %).  Here lane p owns pair p: its logit row Z_p[0..KD) lives in KD registers and the row of W for
// the current k is a broadcast LDS.128 shared by all lanes: per 4 k, 2 + 16 LDS.128 and 4 FMUL feed 256 FMA.  The pair
// products are formed on the fly from the sample's F embedding rows (row stride KD+4: conflict-free for LDS.128 with one
// row per lane, and for scalar access with lanes over k).  dP_p = a_p d_afm + dZ_p W^T has the same shape (W^T is kept in
// shared memory too) and is written in place over dZ_p.  A round whose tail has <= 16 pairs splits the columns between the
// two half-warps instead of idling half the lanes (P = 45: 1.5 rounds, not 2).
// Per tile of NW samples:  phase A (forward, dZ) | barrier | dW sweep over the tile (warp owns 2 KD/NW columns of half the
// tile's samples, lanes over k) | barrier | phase B (dP over dZ, dE, scatter).  Shared memory per warp is F + P rows, so 8 warps (2 per scheduler)
// fit next to W and W^T.
// ---------------------------------------------------------------------------------------------------------------
__host__ __device__ inline int afm2_p4(int P) { return (P + 3) / 4 * 4; }
__host__ __device__ inline size_t afm2_per_warp_floats(int F, int KD, int P, bool drop = false) {
  return (size_t)F * KD + KD + (drop ? 3 : 2) * (size_t)afm2_p4(P) + (size_t)(F + P) * (KD + 4);   // every term a multiple of 4
}
__host__ __device__ inline size_t afm2_smem_floats(int NW, int F, int KD, int P, bool drop = false) {
  return 2 * (size_t)KD * KD + 3 * (size_t)KD + (size_t)NW * afm2_per_warp_floats(F, KD, P, drop) + 32;
}

// acc[r][c] += sum_k x_rk * Wc[k*KD + c], c in [0, NC), r in [0, NR), with x_rk = u_r[k] * v_r[k] (PROD) or u_r[k].
// One broadcast LDS.128 of W (2 shared-memory wavefronts for 16 bytes - the cost that bounds this kernel) feeds 4*NR FMAs.
template <int KD, int NC, int NR, bool PROD>
__device__ __forceinline__ void afm2_rows_times_matrix(float (&acc)[NR][NC], const float* const (&u)[NR], const float* const (&v)[NR],
                                                       const float* __restrict__ Wc) {
#pragma unroll 1
  for (int k = 0; k < KD; k += 4) {
    float x[NR][4];
#pragma unroll
    for (int r = 0; r < NR; r++) {
      const float4 x4 = *reinterpret_cast<const float4*>(u[r] + k);
      x[r][0] = x4.x; x[r][1] = x4.y; x[r][2] = x4.z; x[r][3] = x4.w;
      if (PROD) {
        const float4 y4 = *reinterpret_cast<const float4*>(v[r] + k);
        x[r][0] *= y4.x; x[r][1] *= y4.y; x[r][2] *= y4.z; x[r][3] *= y4.w;
      }
    }
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
      const float4* w4 = reinterpret_cast<const float4*>(Wc + (k + kk) * KD);
#pragma unroll
      for (int c4 = 0; c4 < NC / 4; c4++) {
        const float4 w = w4[c4];
#pragma unroll
        for (int r = 0; r < NR; r++) {
          acc[r][4 * c4] = fmaf(x[r][kk], w.x, acc[r][4 * c4]);
          acc[r][4 * c4 + 1] = fmaf(x[r][kk], w.y, acc[r][4 * c4 + 1]);
          acc[r][4 * c4 + 2] = fmaf(x[r][kk], w.z, acc[r][4 * c4 + 2]);
          acc[r][4 * c4 + 3] = fmaf(x[r][kk], w.w, acc[r][4 * c4 + 3]);
        }
      }
    }
  }
}

// Lane (h, l) = (lane >> 4, lane & 15) owns pairs l, l + 16, ... (NR of them) and the column half [h*KD/2, (h+1)*KD/2).
// Logits: Z_p = P_p W + b into sZ, s_p = relu(Z_p) . p into sS.
template <int KD, int NR>
__device__ __forceinline__ void afm2_logits(const float* sE, const unsigned char* sPairI, const unsigned char* sPairJ, const float* sW,
                                            const float* sb, const float* sp, float* sZ, float* sS, int P, int lane) {
  constexpr int NC = KD / 2, RS = KD + 4;
  const int c0 = (lane >> 4) * NC, l = lane & 15;
  float acc[NR][NC];
  const float* u[NR]; const float* v[NR];
#pragma unroll
  for (int r = 0; r < NR; r++) {
    const int p = l + 16 * r, q = p < P ? p : 0;
    u[r] = sE + sPairI[q] * RS; v[r] = sE + sPairJ[q] * RS;
#pragma unroll
    for (int c = 0; c < NC; c++) acc[r][c] = sb[c0 + c];
  }
  afm2_rows_times_matrix<KD, NC, NR, true>(acc, u, v, sW + c0);
#pragma unroll
  for (int r = 0; r < NR; r++) {
    const int p = l + 16 * r;
    float sc = 0.f;
#pragma unroll
    for (int c = 0; c < NC; c++) sc = fmaf(fmaxf(acc[r][c], 0.f), sp[c0 + c], sc);
    sc += __shfl_xor_sync(0xffffffffu, sc, 16);
    if (p < P) {
#pragma unroll
      for (int c4 = 0; c4 < NC / 4; c4++)
        reinterpret_cast<float4*>(sZ + p * RS + c0)[c4] = make_float4(acc[r][4 * c4], acc[r][4 * c4 + 1], acc[r][4 * c4 + 2], acc[r][4 * c4 + 3]);
      if (lane < 16) sS[p] = sc;
    }
  }
}

// dP_p = a_p d_afm + dZ_p W^T, written over dZ_p (both lanes of a row finish reading it before either writes);
// DROP: a_p m_p d_afm, m_p from sM
template <int KD, int NR, bool DROP = false>
__device__ __forceinline__ void afm2_dpairs(float* sZ, const float* sWT, const float* sdafm, const float* sS, const float* sM, int P,
                                            int lane) {
  constexpr int NC = KD / 2, RS = KD + 4;
  const int c0 = (lane >> 4) * NC, l = lane & 15;
  float acc[NR][NC];
  const float* u[NR];
#pragma unroll
  for (int r = 0; r < NR; r++) {
    const int p = l + 16 * r;
    const float ap = p < P ? (DROP ? sS[p] * sM[p] : sS[p]) : 0.f;
    u[r] = sZ + (p < P ? p : 0) * RS;
#pragma unroll
    for (int c = 0; c < NC; c++) acc[r][c] = ap * sdafm[c0 + c];
  }
  afm2_rows_times_matrix<KD, NC, NR, false>(acc, u, u, sWT + c0);
  __syncwarp();
#pragma unroll
  for (int r = 0; r < NR; r++) {
    const int p = l + 16 * r;
    if (p < P) {
#pragma unroll
      for (int c4 = 0; c4 < NC / 4; c4++)
        reinterpret_cast<float4*>(sZ + p * RS + c0)[c4] = make_float4(acc[r][4 * c4], acc[r][4 * c4 + 1], acc[r][4 * c4 + 2], acc[r][4 * c4 + 3]);
    }
  }
}

// DROP: training dropout, as in afm_kernel
template <int KD, int NW, int NR, bool TRAIN, bool DROP = false>
__global__ void __launch_bounds__(NW * 32, 1) afm2_kernel(const AfmArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float scratch[32];
  __shared__ unsigned char sPairI[kAfmMaxP], sPairJ[kAfmMaxP];
  constexpr int RS = KD + 4;                 // row stride of sE / sZ
  constexpr int TD = (KD + 31) / 32;         // values per lane when the lanes run over k / a
  constexpr int SG = (NW >= 8 && KD >= 32) ? 2 : 1;   // the tile's samples are split over SG groups of warps for the dW sweep
  constexpr int AS = KD * SG / NW;           // columns of dW per warp (more columns per warp = more FMAs per loaded operand)
  static_assert(AS % 4 == 0, "dW column slice is read with LDS.128");
  const int F = a.F, P = a.P, P4 = afm2_p4(P);
  float* sW = smem;                          // [KD][KD]   W[k][a]
  float* sWT = sW + KD * KD;                 // [KD][KD]   W^T[a][k]
  float* sp = sWT + KD * KD;                 // [KD]
  float* sb = sp + KD;                       // [KD]
  float* swp = sb + KD;                      // [KD]
  float* warp_base = swp + KD;
  const size_t per_warp = afm2_per_warp_floats(F, KD, P, DROP);
  int* sValid = reinterpret_cast<int*>(warp_base + (size_t)NW * per_warp);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sDE = warp_base + warp * per_warp;  // [F][KD]
  float* sdafm = sDE + (size_t)F * KD;       // [KD]
  float* sS = sdafm + KD;                    // [P] s, later a
  float* sD = sS + P4;                       // [P] d a, later d s
  float* sM = sD + P4;                       // [P] m_p (DROP only)
  float* sE = sM + (DROP ? P4 : 0);          // [F][RS]
  float* sZ = sE + (size_t)F * RS;           // [P][RS]  Z, then dZ, then dP
  const size_t offE = (size_t)F * KD + KD + (DROP ? 3 : 2) * (size_t)P4;
  const uint64_t vseed = DROP ? splitmix64(a.drop_seed) : 0;

  for (int i = threadIdx.x; i < KD * KD; i += blockDim.x) {
    const float w = __ldg(a.W + i);
    sW[i] = w;
    sWT[(i % KD) * KD + (i / KD)] = w;
  }
  for (int i = threadIdx.x; i < KD; i += blockDim.x) { sp[i] = __ldg(a.pvec + i); sb[i] = __ldg(a.batt + i); swp[i] = __ldg(a.wpred + i); }
  if (threadIdx.x == 0) {
    int p = 0;
    for (int i = 0; i < F; i++)
      for (int j = i + 1; j < F; j++) { sPairI[p] = (unsigned char)i; sPairJ[p] = (unsigned char)j; p++; }
  }
  __syncthreads();

  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  const int rep = a.hot.slot ? (int)(((int64_t)blockIdx.x * NW + warp) % a.hot.n_rep) : 0;
  float dWacc[TRAIN ? TD : 1][AS];
  float gbatt_acc[TD], gp_acc[TD], gwp_acc[TD];
  float loss_acc = 0.f, g0_acc = 0.f;
  if (TRAIN) {
#pragma unroll
    for (int t = 0; t < TD; t++)
#pragma unroll
      for (int r = 0; r < AS; r++) dWacc[t][r] = 0.f;
  }
#pragma unroll
  for (int t = 0; t < TD; t++) { gbatt_acc[t] = 0.f; gp_acc[t] = 0.f; gwp_acc[t] = 0.f; }

  for (int64_t s0 = (int64_t)blockIdx.x * NW; s0 < a.B; s0 += (int64_t)gridDim.x * NW) {
    const int64_t s = s0 + warp;
    const bool valid = s < a.B;
    float g = 0.f;
    if (lane == 0) sValid[warp] = valid ? 1 : 0;
    if (valid) {
      const int32_t* rec = a.idx + s * F;
      // ---- gather E and the bias sum ----
      float bsum = 0.f;
      for (int f = 0; f < F; f++) {
        const int id = __ldg(rec + f);
        for (int k = lane; k < KD; k += 32) sE[f * RS + k] = __ldg(a.V + (size_t)id * KD + k);
        if (a.bias) bsum += __ldg(a.bias + id);
      }
      __syncwarp();
      // ---- logits: lane = (column half, pair mod 16) ----
      afm2_logits<KD, NR>(sE, sPairI, sPairJ, sW, sb, sp, sZ, sS, P, lane);
      __syncwarp();
      // ---- softmax over pairs (AFM.py:125) ----
      float mx = -INFINITY;
      for (int p = lane; p < P; p += 32) mx = fmaxf(mx, sS[p]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float den = 0.f;
      for (int p = lane; p < P; p += 32) { const float e = expf(sS[p] - mx); sS[p] = e; den += e; }
      den = warp_sum(den);
      __syncwarp();
      for (int p = lane; p < P; p += 32) {
        sS[p] = sS[p] / den;
        if (DROP) sM[p] = afm_mask_att(a, s, p) / a.keep_att;
      }
      __syncwarp();
      float nv[TD];                                               // n_k of the lane's columns (DROP)
#pragma unroll
      for (int t = 0; t < TD; t++) nv[t] = DROP ? afm_mask_vec(a, vseed, s, lane + 32 * t) / a.keep_vec : 1.f;
      // ---- afm = sum_p a_p E_i E_j (lanes over k), out ----
      float afm[TD];
#pragma unroll
      for (int t = 0; t < TD; t++) afm[t] = 0.f;
      {
        int p = 0;
        for (int i = 0; i < F; i++) {
          float ei[TD], in[TD];
#pragma unroll
          for (int t = 0; t < TD; t++) { const int k = lane + 32 * t; ei[t] = (k < KD) ? sE[i * RS + k] : 0.f; in[t] = 0.f; }
          for (int j = i + 1; j < F; j++, p++) {
            const float ap = DROP ? sS[p] * sM[p] : sS[p];
#pragma unroll
            for (int t = 0; t < TD; t++) { const int k = lane + 32 * t; if (k < KD) in[t] = fmaf(ap, sE[j * RS + k], in[t]); }
          }
#pragma unroll
          for (int t = 0; t < TD; t++) afm[t] = fmaf(ei[t], in[t], afm[t]);
        }
      }
      float part = 0.f;
#pragma unroll
      for (int t = 0; t < TD; t++) { const int k = lane + 32 * t; if (k < KD) part = fmaf(afm[t], DROP ? swp[k] * nv[t] : swp[k], part); }
      const float bil = warp_sum(part);
      const float out = (bil + bsum) + b0;                       // AFM.py:142 add_n
      if (a.out && lane == 0) a.out[s] = out;

      if (TRAIN) {
        const float y = __ldg(a.labels + s);
        const float diff = y - out;
        g = -diff;
        if (lane == 0) { loss_acc += 0.5f * diff * diff; g0_acc += g; }
#pragma unroll
        for (int t = 0; t < TD; t++) {
          const int k = lane + 32 * t;
          if (k < KD) {
            sdafm[k] = g * (DROP ? swp[k] * nv[t] : swp[k]);
            gwp_acc[t] = fmaf(g, DROP ? afm[t] * nv[t] : afm[t], gwp_acc[t]);
          }
        }
        __syncwarp();
        // ---- d a_p = (E_i E_j) . d afm (lane = pair), softmax backward ----
        float dotp = 0.f;
        for (int p = lane; p < P; p += 32) {
          const float* ei = sE + sPairI[p] * RS; const float* ej = sE + sPairJ[p] * RS;
          float v = 0.f;
#pragma unroll 4
          for (int k = 0; k < KD; k += 4) {
            const float4 x = *reinterpret_cast<const float4*>(ei + k), y4 = *reinterpret_cast<const float4*>(ej + k);
            const float4 d = *reinterpret_cast<const float4*>(sdafm + k);
            v = fmaf(x.x * y4.x, d.x, v); v = fmaf(x.y * y4.y, d.y, v); v = fmaf(x.z * y4.z, d.z, v); v = fmaf(x.w * y4.w, d.w, v);
          }
          sD[p] = v;
          dotp = fmaf(DROP ? sS[p] * sM[p] : sS[p], v, dotp);
        }
        const float dot = warp_sum(dotp);
        __syncwarp();
        for (int p = lane; p < P; p += 32) sD[p] = sS[p] * ((DROP ? sM[p] * sD[p] : sD[p]) - dot);       // d s_p
        __syncwarp();
        // ---- d Z_p = d s_p p (Z_p > 0) (over Z) ; d p += d s_p relu(Z_p) ; d b += d Z_p  (lanes over a) ----
        for (int p = 0; p < P; p++) {
          const float ds = sD[p];
#pragma unroll
          for (int t = 0; t < TD; t++) {
            const int aa = lane + 32 * t;
            if (aa < KD) {
              const float z = sZ[p * RS + aa];
              const float dz = (z > 0.f) ? ds * sp[aa] : 0.f;
              gp_acc[t] = fmaf(ds, fmaxf(z, 0.f), gp_acc[t]);
              gbatt_acc[t] += dz;
              sZ[p * RS + aa] = dz;
            }
          }
        }
      }
    }
    if (TRAIN) {
      __syncthreads();
      // ---- d W[k][a] += (E_i E_j)[k] dZ_p[a]: lanes over k; the warps form SG groups, group g sweeps the samples of its
      // share of the tile and warp w of a group owns AS columns (32 FMAs per pair of operand loads instead of 16) ----
      for (int ws = (warp * SG / NW) * (NW / SG); ws < (warp * SG / NW + 1) * (NW / SG); ws++) {
        if (!sValid[ws]) continue;
        const float* oE = warp_base + ws * per_warp + offE;
        const float* oZ = oE + (size_t)F * RS + (warp % (NW / SG)) * AS;
        int p = 0;
        for (int i = 0; i < F; i++) {
          float ei[TD];
#pragma unroll
          for (int t = 0; t < TD; t++) { const int k = lane + 32 * t; ei[t] = (k < KD) ? oE[i * RS + k] : 0.f; }
          for (int j = i + 1; j < F; j++, p++) {
            float pk[TD];
#pragma unroll
            for (int t = 0; t < TD; t++) { const int k = lane + 32 * t; pk[t] = (k < KD) ? ei[t] * oE[j * RS + k] : 0.f; }
#pragma unroll
            for (int r4 = 0; r4 < AS / 4; r4++) {
              const float4 dz = *reinterpret_cast<const float4*>(oZ + p * RS + 4 * r4);
#pragma unroll
              for (int t = 0; t < TD; t++) {
                dWacc[t][4 * r4] = fmaf(pk[t], dz.x, dWacc[t][4 * r4]);
                dWacc[t][4 * r4 + 1] = fmaf(pk[t], dz.y, dWacc[t][4 * r4 + 1]);
                dWacc[t][4 * r4 + 2] = fmaf(pk[t], dz.z, dWacc[t][4 * r4 + 2]);
                dWacc[t][4 * r4 + 3] = fmaf(pk[t], dz.w, dWacc[t][4 * r4 + 3]);
              }
            }
          }
        }
      }
      __syncthreads();
      if (valid) {
        const int32_t* rec = a.idx + s * F;
        // ---- d P_p = a_p d afm + d Z_p W^T, in place ----
        afm2_dpairs<KD, NR, DROP>(sZ, sWT, sdafm, sS, sM, P, lane);
        __syncwarp();
        // ---- d E_f = sum_{g != f} dP_{fg} * E_g  (lanes over k, registers; no read-modify-write through shared memory) ----
        for (int f = 0; f < F; f++) {
          float de[TD];
#pragma unroll
          for (int t = 0; t < TD; t++) de[t] = 0.f;
          for (int o = 0; o < F; o++) {
            if (o == f) continue;
            const int i = f < o ? f : o, j = f < o ? o : f;
            const int p = i * F - ((i * (i + 1)) >> 1) + (j - i - 1);
#pragma unroll
            for (int t = 0; t < TD; t++) {
              const int k = lane + 32 * t;
              if (k < KD) de[t] = fmaf(sZ[p * RS + k], sE[o * RS + k], de[t]);
            }
          }
#pragma unroll
          for (int t = 0; t < TD; t++) { const int k = lane + 32 * t; if (k < KD) sDE[f * KD + k] = de[t]; }
        }
        __syncwarp();
        for (int f = 0; f < F; f++) {
          const int id = __ldg(rec + f);
          float* dst = a.gV + (size_t)id * KD;
          if (a.hot.slot != nullptr) {
            const int hs = __ldg(a.hot.slot + id);
            if (hs >= 0) dst = a.hot.ghot + ((size_t)rep * a.hot.n_hot + hs) * KD;
          }
          for (int c = lane; c < (KD >> 2); c += 32) red_add_v4(dst + 4 * c, reinterpret_cast<const float4*>(sDE + f * KD)[c]);
          if (lane == 0) {
            if (a.gbias) scatter_bias(a.gbias, a.hot, rep, id, g);
            touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, id);
          }
        }
        __syncwarp();
      }
    }
  }

  if (TRAIN) {
#pragma unroll
    for (int t = 0; t < TD; t++) {
      const int k = lane + 32 * t;
      if (k < KD) {
#pragma unroll
        for (int r = 0; r < AS; r++)
          if (dWacc[t][r] != 0.f) atomicAdd(a.gW + (size_t)k * KD + (warp % (NW / SG)) * AS + r, dWacc[t][r]);
        atomicAdd(a.gbatt + k, gbatt_acc[t]); atomicAdd(a.gp + k, gp_acc[t]); atomicAdd(a.gwpred + k, gwp_acc[t]);
      }
    }
    const float bl = block_sum(loss_acc, scratch);
    write_partial(a.loss_partials, bl);
    const float bg = block_sum(g0_acc, scratch);
    if (threadIdx.x == 0 && a.gb0 && bg != 0.f) atomicAdd(a.gb0, bg);
  }
}

template <int KD, int NW, int NR, bool TRAIN, bool DROP>
static int launch_afm2(const AfmArgs& a, cudaStream_t st) {
  const size_t smem = afm2_smem_floats(NW, a.F, KD, a.P, DROP) * sizeof(float);
  if (smem > 220 * 1024) return 1;
  auto kern = afm2_kernel<KD, NW, NR, TRAIN, DROP>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    set_error("afm2_kernel: cannot reserve %zu bytes of shared memory", smem);
    return HHFM_ERR_LAUNCH;
  }
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NW * 32, smem);
  if (occ < 1) occ = 1;
  int64_t need = (a.B + NW - 1) / NW;
  int64_t cap = (int64_t)sm_count() * occ;
  if (cap > kPartials) cap = kPartials;
  const int grid = (int)(need < cap ? need : cap);
  kern<<<grid, NW * 32, smem, st>>>(a);
  return check_launch("afm2_kernel");
}

template <int KD, int NR, bool TRAIN, bool DROP>
static int launch_afm2_warps(const AfmArgs& a, cudaStream_t st) {
  if constexpr (KD >= 32) {
    const int rc = launch_afm2<KD, 8, NR, TRAIN, DROP>(a, st);
    if (rc != 1) return rc;
  }
  return launch_afm2<KD, 4, NR, TRAIN, DROP>(a, st);
}

// returns 1 when the shape is not covered (the caller then uses afm_kernel)
template <bool TRAIN, bool DROP>
static int dispatch_afm2(const AfmArgs& a, cudaStream_t st) {
  const char* e = getenv("HHFM_AFM_V1");           // 1 = force the first layout (A/B measurements, tests of both kernels)
  if (e && e[0] == '1') return 1;
  if (a.K != a.A) return 1;
  const int nr = (a.P + 15) / 16;                   // pairs per lane
  if (nr > 3) return 1;
#define HHFM_AFM2_CASE(KD_)                                                       \
  if (a.K == KD_) {                                                               \
    if (nr == 1) return launch_afm2_warps<KD_, 1, TRAIN, DROP>(a, st);            \
    if (nr == 2) return launch_afm2_warps<KD_, 2, TRAIN, DROP>(a, st);            \
    return launch_afm2_warps<KD_, 3, TRAIN, DROP>(a, st);                         \
  }
  HHFM_AFM2_CASE(64)
  HHFM_AFM2_CASE(32)
  HHFM_AFM2_CASE(16)
#undef HHFM_AFM2_CASE
  return 1;
}

template <int TK, int TA, int NW, bool TRAIN, bool DROP>
static int launch_afm(const AfmArgs& a, cudaStream_t st) {
  const size_t smem = afm_smem_floats(NW, a.F, a.K, a.A, a.P, DROP) * sizeof(float);
  if (smem > 220 * 1024) return 1;
  auto kern = afm_kernel<TK, TA, NW, TRAIN, DROP>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    set_error("afm_kernel: cannot reserve %zu bytes of shared memory", smem);
    return HHFM_ERR_LAUNCH;
  }
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NW * 32, smem);
  if (occ < 1) occ = 1;
  int64_t need = (a.B + NW - 1) / NW;
  int64_t cap = (int64_t)sm_count() * occ;
  if (cap > kPartials) cap = kPartials;
  const int grid = (int)(need < cap ? need : cap);
  kern<<<grid, NW * 32, smem, st>>>(a);
  return check_launch("afm_kernel");
}

// DROP: the training-dropout instantiations (TRAIN only)
template <bool TRAIN, bool DROP = false>
static int dispatch_afm(const AfmArgs& a, cudaStream_t st) {
  {
    const int rc2 = dispatch_afm2<TRAIN, DROP>(a, st);
    if (rc2 != 1) return rc2;
  }
  // largest warp count whose shared-memory footprint fits; K % NW == 0 and K/NW % 4 == 0 are needed by the dW sweep
  const int tk = (a.K + 31) / 32, ta = (a.A + 31) / 32;
  int rc = 1;
#define TRY(TKV, TAV, NWV)                                                      \
  if (rc == 1 && tk == TKV && ta == TAV && a.K % (NWV * 4) == 0) rc = launch_afm<TKV, TAV, NWV, TRAIN, DROP>(a, st);
  TRY(1, 1, 4) TRY(1, 1, 2) TRY(2, 2, 4) TRY(2, 2, 2) TRY(4, 4, 4) TRY(4, 4, 2) TRY(4, 4, 1)
#undef TRY
  if (rc == 1) {
    set_error("afm: configuration F=%d K=%d A=%d does not fit (need K,A in {<=32,<=64,<=128} with equal tiers, shared memory <= 220 KB)",
              a.F, a.K, a.A);
    return HHFM_ERR_UNSUPPORTED;
  }
  return rc;
}

// ---------------------------------------------------------------------------------------------------------------
// attention = 0 (AFM.py:132): afm = sum_p P_p = 0.5 (S^2 - sum_f E_f^2) with S = sum_f E_f, out = (afm n) . prediction_W
// + sum_f bias[x_f] + b0 -- FM's interaction weighted by w~ = prediction_W n (n = the pooled-vector dropout factors, 1 outside
// training).  No attention net, so no shared memory: one warp per sample, lane c owns the float4 chunk c of a row (K <= 128).
// Training: dE_f = g w~ (S - E_f) into the gradient rows (vector reductions, hot-row replicas, touched rows as in afm_kernel),
// d prediction_W += g n afm in registers, one atomic per column at the end.
// ---------------------------------------------------------------------------------------------------------------
template <bool TRAIN>
__global__ void __launch_bounds__(kBlock) afm_sum_kernel(const AfmArgs a) {
  __shared__ float scratch[32];
  constexpr int NW = kBlock / 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = a.F, K = a.K;
  const bool on = lane < (K >> 2);
  const bool drop = TRAIN && a.keep_vec < 1.f;
  const uint64_t vseed = splitmix64(a.drop_seed);
  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  const float4 wp = on ? __ldg(reinterpret_cast<const float4*>(a.wpred) + lane) : f4_zero();
  const int rep = a.hot.slot ? (int)(((int64_t)blockIdx.x * NW + warp) % a.hot.n_rep) : 0;
  float4 gwp_acc = f4_zero();
  float loss_acc = 0.f, g0_acc = 0.f;
  for (int64_t s = (int64_t)blockIdx.x * NW + warp; s < a.B; s += (int64_t)gridDim.x * NW) {
    const int32_t* rec = a.idx + s * F;
    float4 S = f4_zero(), Q = f4_zero();
    float bsum = 0.f;
    for (int f = 0; f < F; f++) {
      const int id = __ldg(rec + f);
      if (on) {
        const float4 e = __ldg(reinterpret_cast<const float4*>(a.V + (size_t)id * K) + lane);
        S = f4_add(S, e);
        Q = f4_add(Q, f4_mul(e, e));
      }
      if (a.bias) bsum += __ldg(a.bias + id);
    }
    float4 n = make_float4(1.f, 1.f, 1.f, 1.f);
    if (drop && on)
      n = make_float4(afm_mask_vec(a, vseed, s, 4 * lane) / a.keep_vec, afm_mask_vec(a, vseed, s, 4 * lane + 1) / a.keep_vec,
                      afm_mask_vec(a, vseed, s, 4 * lane + 2) / a.keep_vec, afm_mask_vec(a, vseed, s, 4 * lane + 3) / a.keep_vec);
    const float4 afm = f4_scale(f4_sub(f4_mul(S, S), Q), 0.5f);
    const float4 wt = f4_mul(wp, n);                                    // w~ (zero on the lanes past K)
    const float out = (warp_sum(f4_dot(afm, wt)) + bsum) + b0;
    if (a.out && lane == 0) a.out[s] = out;
    if (TRAIN) {
      const float diff = __ldg(a.labels + s) - out;
      const float g = -diff;
      if (lane == 0) { loss_acc += 0.5f * diff * diff; g0_acc += g; }
      gwp_acc = f4_fma(f4_mul(afm, n), g, gwp_acc);
      const float4 dt = f4_scale(wt, g);
      for (int f = 0; f < F; f++) {
        const int id = __ldg(rec + f);
        if (on) {
          float* dst = a.gV + (size_t)id * K;
          if (a.hot.slot != nullptr) {
            const int hs = __ldg(a.hot.slot + id);
            if (hs >= 0) dst = a.hot.ghot + ((size_t)rep * a.hot.n_hot + hs) * K;
          }
          const float4 e = __ldg(reinterpret_cast<const float4*>(a.V + (size_t)id * K) + lane);
          red_add_v4(dst + 4 * lane, f4_mul(dt, f4_sub(S, e)));
        }
        if (lane == 0) {
          if (a.gbias) scatter_bias(a.gbias, a.hot, rep, id, g);
          touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, id);
        }
      }
    }
  }
  if (TRAIN) {
    if (on) {
      atomicAdd(a.gwpred + 4 * lane, gwp_acc.x); atomicAdd(a.gwpred + 4 * lane + 1, gwp_acc.y);
      atomicAdd(a.gwpred + 4 * lane + 2, gwp_acc.z); atomicAdd(a.gwpred + 4 * lane + 3, gwp_acc.w);
    }
    const float bl = block_sum(loss_acc, scratch);
    write_partial(a.loss_partials, bl);
    const float bg = block_sum(g0_acc, scratch);
    if (threadIdx.x == 0 && a.gb0 && bg != 0.f) atomicAdd(a.gb0, bg);
  }
}

template <bool TRAIN>
static int launch_afm_sum(const AfmArgs& a, cudaStream_t st) {
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, afm_sum_kernel<TRAIN>, kBlock, 0);
  if (occ < 1) occ = 1;
  afm_sum_kernel<TRAIN><<<grid_for(a.B, kBlock / 32, occ), kBlock, 0, st>>>(a);
  return check_launch("afm_sum_kernel");
}

static int check_afm(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* W, const float* batt,
                     const float* pvec, const float* wpred, int64_t M, int64_t K, int64_t A) {
  HHFM_REQUIRE(idx && V && W && batt && pvec && wpred, "afm: NULL argument");
  HHFM_REQUIRE(B >= 0 && M > 0, "afm: bad sizes");
  HHFM_REQUIRE(F >= 2 && F <= kAfmMaxF, "afm: F=%lld out of range [2,%d]", (long long)F, kAfmMaxF);
  HHFM_REQUIRE(K % 4 == 0 && K >= 4 && K <= 128 && A % 4 == 0 && A >= 4 && A <= 128, "afm: K=%lld A=%lld unsupported (multiples of 4, <= 128)",
               (long long)K, (long long)A);
  HHFM_REQUIRE(((uintptr_t)V & 15) == 0, "afm: V must be 16-byte aligned");
  return HHFM_OK;
}

static AfmArgs make_afm(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias, const float* b0,
                        const float* W, const float* batt, const float* pvec, const float* wpred, int64_t K, int64_t A) {
  AfmArgs a{};
  a.idx = idx; a.B = B; a.F = (int)F; a.K = (int)K; a.A = (int)A; a.P = (int)(F * (F - 1) / 2);
  a.V = V; a.bias = bias; a.b0 = b0; a.W = W; a.batt = batt; a.pvec = pvec; a.wpred = wpred;
  return a;
}

static int make_afm_train(AfmArgs& a, const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias, const float* b0,
                          const float* W, const float* batt, const float* pvec, const float* wpred, int64_t M, int64_t K, int64_t A,
                          const float* labels, float* out, float* gV, float* gbias, float* gb0, float* gW, float* gbatt, float* gp,
                          float* gwpred, float* loss_partials, int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows,
                          int32_t* touched_count, const int32_t* hot_slot, float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot) {
  int rc = check_afm(idx, B, F, V, W, batt, pvec, wpred, M, K, A);
  if (rc) return rc;
  HHFM_REQUIRE(B > 0 && labels && gV && gW && gbatt && gp && gwpred && loss_partials, "afm_fwd_bwd_sqloss: NULL argument");
  HHFM_REQUIRE(!touch_stamp || (touched_rows && touched_count), "afm_fwd_bwd_sqloss: touch_stamp needs touched_rows/count");
  HHFM_REQUIRE(!hot_slot || (ghot && n_rep >= 1 && n_hot >= 1), "afm_fwd_bwd_sqloss: hot_slot needs ghot, n_rep, n_hot");
  a = make_afm(idx, B, F, V, bias, b0, W, batt, pvec, wpred, K, A);
  a.labels = labels; a.out = out; a.gV = gV; a.gbias = gbias; a.gb0 = gb0; a.gW = gW; a.gbatt = gbatt; a.gp = gp;
  a.gwpred = gwpred; a.loss_partials = loss_partials; a.touch_stamp = touch_stamp; a.stamp = stamp;
  a.touched_rows = touched_rows; a.touched_count = touched_count;
  a.hot = HotPlan{hot_slot, ghot, ghot_bias, n_rep, n_hot};
  return HHFM_OK;
}

}  // namespace hhfm

using namespace hhfm;

extern "C" int hhfm_afm_fwd(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias, const float* b0,
                            const float* W, const float* batt, const float* pvec, const float* wpred, int64_t M, int64_t K,
                            int64_t A, float* out, hhfm_stream_t stream) {
  int rc = check_afm(idx, B, F, V, W, batt, pvec, wpred, M, K, A);
  if (rc) return rc;
  HHFM_REQUIRE(out != nullptr, "afm_fwd: out is NULL");
  if (B == 0) return HHFM_OK;
  AfmArgs a = make_afm(idx, B, F, V, bias, b0, W, batt, pvec, wpred, K, A);
  a.out = out;
  return dispatch_afm<false>(a, (cudaStream_t)stream);
}

extern "C" int hhfm_afm_fwd_attn(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias, const float* b0,
                                 const float* W, const float* batt, const float* pvec, const float* wpred, int64_t M, int64_t K,
                                 int64_t A, int32_t attention, float* out, hhfm_stream_t stream) {
  HHFM_REQUIRE(attention == 0 || attention == 1, "afm_fwd_attn: attention=%d must be 0 or 1", (int)attention);
  if (attention == 1) return hhfm_afm_fwd(idx, B, F, V, bias, b0, W, batt, pvec, wpred, M, K, A, out, stream);
  int rc = check_afm(idx, B, F, V, W, batt, pvec, wpred, M, K, A);
  if (rc) return rc;
  HHFM_REQUIRE(out != nullptr, "afm_fwd_attn: out is NULL");
  HHFM_REQUIRE(((uintptr_t)wpred & 15) == 0, "afm: prediction_W must be 16-byte aligned");
  if (B == 0) return HHFM_OK;
  AfmArgs a = make_afm(idx, B, F, V, bias, b0, W, batt, pvec, wpred, K, A);
  a.out = out;
  return launch_afm_sum<false>(a, (cudaStream_t)stream);
}

extern "C" int hhfm_afm_fwd_bwd_sqloss(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias,
                                       const float* b0, const float* W, const float* batt, const float* pvec,
                                       const float* wpred, int64_t M, int64_t K, int64_t A, const float* labels, float* out,
                                       float* gV, float* gbias, float* gb0, float* gW, float* gbatt, float* gp, float* gwpred,
                                       float* loss_partials, int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows,
                                       int32_t* touched_count, const int32_t* hot_slot, float* ghot, float* ghot_bias,
                                       int32_t n_rep, int32_t n_hot, hhfm_stream_t stream) {
  AfmArgs a;
  int rc = make_afm_train(a, idx, B, F, V, bias, b0, W, batt, pvec, wpred, M, K, A, labels, out, gV, gbias, gb0, gW, gbatt, gp,
                          gwpred, loss_partials, touch_stamp, stamp, touched_rows, touched_count, hot_slot, ghot, ghot_bias, n_rep,
                          n_hot);
  if (rc) return rc;
  {
    const int frc = dispatch_afm_fused_tc(a, M, (cudaStream_t)stream);      // K = A = 64, F <= 11: one tcgen05 kernel
    if (frc != 1) return frc;
  }
  return dispatch_afm<true>(a, (cudaStream_t)stream);
}

extern "C" int hhfm_afm_fwd_bwd_sqloss_dropout(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias,
                                               const float* b0, const float* W, const float* batt, const float* pvec,
                                               const float* wpred, int64_t M, int64_t K, int64_t A, const float* labels,
                                               float* out, float* gV, float* gbias, float* gb0, float* gW, float* gbatt, float* gp,
                                               float* gwpred, float* loss_partials, int32_t* touch_stamp, int32_t stamp,
                                               int32_t* touched_rows, int32_t* touched_count, const int32_t* hot_slot,
                                               float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot, int32_t attention,
                                               float keep_att, float keep_vec, uint64_t drop_seed, int64_t sample_base,
                                               hhfm_stream_t stream) {
  HHFM_REQUIRE(attention == 0 || attention == 1, "afm_fwd_bwd_sqloss_dropout: attention=%d must be 0 or 1", (int)attention);
  HHFM_REQUIRE(keep_att > 0.f && keep_att <= 1.f && keep_vec > 0.f && keep_vec <= 1.f,
               "afm_fwd_bwd_sqloss_dropout: dropout keep [%g, %g] must be in (0, 1]", (double)keep_att, (double)keep_vec);
  HHFM_REQUIRE(sample_base >= 0, "afm_fwd_bwd_sqloss_dropout: sample_base=%lld must be >= 0", (long long)sample_base);
  const bool drop = keep_att < 1.f || keep_vec < 1.f;
  if (attention == 1 && !drop)                            // keep = [1, 1]: the kernels of hhfm_afm_fwd_bwd_sqloss, unchanged
    return hhfm_afm_fwd_bwd_sqloss(idx, B, F, V, bias, b0, W, batt, pvec, wpred, M, K, A, labels, out, gV, gbias, gb0, gW, gbatt, gp,
                                   gwpred, loss_partials, touch_stamp, stamp, touched_rows, touched_count, hot_slot, ghot, ghot_bias,
                                   n_rep, n_hot, stream);
  AfmArgs a;
  int rc = make_afm_train(a, idx, B, F, V, bias, b0, W, batt, pvec, wpred, M, K, A, labels, out, gV, gbias, gb0, gW, gbatt, gp,
                          gwpred, loss_partials, touch_stamp, stamp, touched_rows, touched_count, hot_slot, ghot, ghot_bias, n_rep,
                          n_hot);
  if (rc) return rc;
  a.keep_att = keep_att; a.keep_vec = keep_vec; a.drop_seed = drop_seed; a.sample_base = sample_base;
  const cudaStream_t st = (cudaStream_t)stream;
  if (attention == 0) {
    HHFM_REQUIRE(((uintptr_t)wpred & 15) == 0, "afm: prediction_W must be 16-byte aligned");
    return launch_afm_sum<true>(a, st);
  }
  {
    const int frc = dispatch_afm_fused_tc(a, M, st, true);
    if (frc != 1) return frc;
  }
  return dispatch_afm<true, true>(a, st);
}
