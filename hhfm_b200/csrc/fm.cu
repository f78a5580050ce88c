// K1: FM / MF gather + second-order interaction, fused with the squared loss and the backward scatter.
// Reference graph: Newcode/FM.py:99-126 (forward + loss), TF autodiff for the backward; MF.py:81-98.
//
// Mapping: one sample is owned by a group of LPS = K/4 lanes (an aligned sub-warp), each lane holding one
// float4 of every embedding row -> every gathered row is one fully coalesced K*4-byte read, the reduction
// over fields is per-lane register work, and only the final sum over k needs log2(LPS) shuffles.
// The backward re-reads the rows (L1/L2 hits) and issues one REDG.E.ADD.F32x4 per 16 bytes.
#include <stdlib.h>

#include "common.cuh"
#include "staged.cuh"

namespace hhfm {

struct FmArgs {
  const int32_t* row_ptr;
  const int32_t* col;
  const float* val;
  int64_t B;
  int F;
  const float* V;
  const float* bias;
  const float* b0;
  int K;
  int interaction;
  const float* labels;
  const float* gout;
  float* out;
  float* gV;
  float* gbias;
  float* gb0;
  float* loss_partials;
  int32_t* touch_stamp;
  int32_t stamp;
  int32_t* touched_rows;
  int32_t* touched_count;
  int groups_active;
  HotPlan hot;
  float keep;            // dropout keep probability of the interaction layer (FM.py:114, MF.py:87); 1 = off
  uint64_t drop_seed;
};

enum { FM_FWD = 0, FM_TRAIN = 1, FM_BWD = 2 };

// DROP: tf.nn.dropout on the [B, K] interaction vector before the sum over k (training launches only; the reference
// evaluates with dropout_keep = 1).  m_k / keep multiplies element k of the vector and of every gradient that flows
// through it.
template <int LPS, int VPL, int MODE, bool DROP = false>
__global__ void __launch_bounds__(kBlock) fm_kernel(const FmArgs a) {
  __shared__ float scratch[32];
  using F4 = Frag<LPS, VPL>;
  const int lane = threadIdx.x & 31, lg = lane % LPS, grp = lane / LPS;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int ga = a.groups_active;
  const int K = a.K;
  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  float loss_acc = 0.f, g0_acc = 0.f;
  const int rep = a.hot.slot ? (int)((warp_g * (32 / LPS) + grp) % a.hot.n_rep) : 0;

  for (int64_t s0 = warp_g * ga; s0 < a.B; s0 += n_warps * ga) {
    const int64_t s = s0 + grp;
    const bool valid = (grp < ga) && (s < a.B);
    int64_t beg = 0, end = 0;
    if (valid) {
      if (a.row_ptr) {
        beg = __ldg(a.row_ptr + s);
        end = __ldg(a.row_ptr + s + 1);
      } else {
        beg = s * a.F;
        end = beg + a.F;
      }
    }
    F4 S, Q, e0, e1, dm;
    frag_zero(S);
    frag_zero(Q);
    frag_zero(e0);
    frag_zero(e1);
    float bsum = 0.f, part = 0.f;
    if (DROP) {
      const int64_t sm = valid ? s : 0;
#pragma unroll
      for (int i = 0; i < VPL; i++) {
        const int k0 = 4 * (lg + i * LPS);
        dm.v[i] = make_float4(dropout_keep01(a.drop_seed, sm, k0, a.keep), dropout_keep01(a.drop_seed, sm, k0 + 1, a.keep),
                              dropout_keep01(a.drop_seed, sm, k0 + 2, a.keep), dropout_keep01(a.drop_seed, sm, k0 + 3, a.keep));
      }
    }

    if (a.interaction == 0) {
      // ---- FM.py:99-109: S = sum_f e_f, Q = sum_f e_f^2 (fields in order, 4 gathers in flight) ----
      for (int64_t j = beg; j < end; j += 4) {
        int id[4];
        float vv[4];
        F4 e[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const bool ok = (j + u) < end;
          id[u] = ok ? __ldg(a.col + j + u) : -1;
          vv[u] = (ok && a.val) ? __ldg(a.val + j + u) : 1.f;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          if (id[u] >= 0) frag_load(e[u], a.V, id[u], K, lg);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          if (id[u] >= 0) {
            if (a.bias) bsum += vv[u] * __ldg(a.bias + id[u]);
#pragma unroll
            for (int i = 0; i < VPL; i++) {
              float4 x = a.val ? f4_scale(e[u].v[i], vv[u]) : e[u].v[i];
              S.v[i] = f4_add(S.v[i], x);
              Q.v[i] = f4_add(Q.v[i], f4_mul(x, x));
            }
          }
        }
      }
#pragma unroll
      for (int i = 0; i < VPL; i++) {
        float4 t = f4_sub(f4_mul(S.v[i], S.v[i]), Q.v[i]);
        if (DROP) {
          t = f4_scale(t, 0.5f);                                   // FM.py:109 `0.5 * subtract`, then :114 dropout
          t = f4_mul(make_float4(t.x / a.keep, t.y / a.keep, t.z / a.keep, t.w / a.keep), dm.v[i]);
          part += f4_hsum(t);
        } else {
          part += 0.5f * f4_hsum(t);
        }
      }
    } else {
      // ---- MF.py:81-92: out = sum_k V[x0]*V[x1]; the bias term is not added (:92) ----
      if (valid) {
        frag_load(e0, a.V, __ldg(a.col + beg), K, lg);
        frag_load(e1, a.V, __ldg(a.col + beg + 1), K, lg);
      }
      if (DROP) {
#pragma unroll
        for (int i = 0; i < VPL; i++) {
          const float4 t = f4_mul(e0.v[i], e1.v[i]);
          part += f4_hsum(f4_mul(make_float4(t.x / a.keep, t.y / a.keep, t.z / a.keep, t.w / a.keep), dm.v[i]));
        }
      } else {
        part = frag_dot(e0, e1);
      }
    }
    const float bil = group_sum<LPS>(part);
    const float out = (bil + bsum) + b0;   // FM.py:120 add_n([Bilinear, Feature_bias, Bias])

    if (MODE == FM_FWD) {
      if (valid && lg == 0) a.out[s] = out;
    }
    float g = 0.f;
    if (MODE == FM_TRAIN) {
      const float y = valid ? __ldg(a.labels + s) : out;
      const float diff = y - out;
      g = -diff;                            // d(0.5*diff^2)/d out
      if (valid && lg == 0) {
        loss_acc += 0.5f * diff * diff;     // FM.py:124 tf.nn.l2_loss
        if (a.out) a.out[s] = out;
      }
    } else if (MODE == FM_BWD) {
      g = valid ? __ldg(a.gout + s) : 0.f;
    }
    if (MODE == FM_FWD || !valid) {
      // nothing to scatter (forward-only launch, or a padding group of the last warp)
    } else {
    if (lg == 0) g0_acc += g;

    // ---- backward: gV[x_f] += g*val_f*(S - e_f); gbias[x_f] += g*val_f ----
    if (a.interaction == 0) {
      for (int64_t j = beg; j < end; j += 4) {
        int id[4];
        float vv[4];
        F4 e[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const bool ok = (j + u) < end;
          id[u] = ok ? __ldg(a.col + j + u) : -1;
          vv[u] = (ok && a.val) ? __ldg(a.val + j + u) : 1.f;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          if (id[u] >= 0) frag_load(e[u], a.V, id[u], K, lg);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          if (id[u] >= 0) {
            const float gv = g * vv[u];
            F4 d;
#pragma unroll
            for (int i = 0; i < VPL; i++) {
              float4 x = a.val ? f4_scale(e[u].v[i], vv[u]) : e[u].v[i];
              d.v[i] = f4_scale(f4_sub(S.v[i], x), gv);
              if (DROP) d.v[i] = f4_mul(d.v[i], make_float4(dm.v[i].x / a.keep, dm.v[i].y / a.keep, dm.v[i].z / a.keep, dm.v[i].w / a.keep));
            }
            scatter_row<LPS, VPL>(a.gV, a.hot, rep, id[u], K, lg, d);
            if (lg == 0) {
              if (a.gbias) scatter_bias(a.gbias, a.hot, rep, id[u], gv);
              touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, id[u]);
            }
          }
        }
      }
    } else {
      const int x0 = __ldg(a.col + beg), x1 = __ldg(a.col + beg + 1);
      F4 d0, d1;
#pragma unroll
      for (int i = 0; i < VPL; i++) {
        d0.v[i] = f4_scale(e1.v[i], g);
        d1.v[i] = f4_scale(e0.v[i], g);
        if (DROP) {
          const float4 mk = make_float4(dm.v[i].x / a.keep, dm.v[i].y / a.keep, dm.v[i].z / a.keep, dm.v[i].w / a.keep);
          d0.v[i] = f4_mul(d0.v[i], mk);
          d1.v[i] = f4_mul(d1.v[i], mk);
        }
      }
      scatter_row<LPS, VPL>(a.gV, a.hot, rep, x0, K, lg, d0);
      scatter_row<LPS, VPL>(a.gV, a.hot, rep, x1, K, lg, d1);
      if (lg == 0) {
        touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, x0);
        touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, x1);
      }
    }
    }  // valid && MODE != FM_FWD
  }

  if (MODE == FM_TRAIN) {
    const float bl = block_sum(loss_acc, scratch);
    write_partial(a.loss_partials, bl);
  }
  if (MODE != FM_FWD && a.gb0 != nullptr) {
    const float bg = block_sum(g0_acc, scratch);
    if (threadIdx.x == 0 && bg != 0.f) atomicAdd(a.gb0, bg);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Specialised training kernel for the common case (fixed-width rows, implicit values 1.0, FM interaction, K = 4*LPS,
// F <= NF <= LPS).  What it changes over fm_kernel, measured on the scaled config (M = 10^7, K = 128: every row comes
// from HBM): the generic kernel keeps 4 gathers in flight per warp and re-reads the rows for the backward, which left
// DRAM at 12 % with every warp in long-scoreboard stalls.  Here all F row gathers (and the hot-slot / bias lookups) of
// a sample are issued back to back, the rows stay in registers for the backward (no re-read), and the touched-row list
// is appended with one warp-aggregated atomic instead of one per row.
template <int LPS, int NF>
__global__ void __launch_bounds__(kBlock, 2) fm_train_fixed_kernel(const FmArgs a) {
  __shared__ float scratch[32];
  constexpr int G = 32 / LPS;
  const int lane = threadIdx.x & 31, lg = lane % LPS, grp = lane / LPS;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int F = a.F;
  constexpr int K = 4 * LPS;
  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  float loss_acc = 0.f, g0_acc = 0.f;
  const int rep = a.hot.slot ? (int)((warp_g * G + grp) % a.hot.n_rep) : 0;
  const float4* V4 = reinterpret_cast<const float4*>(a.V);

  for (int64_t s0 = warp_g * G; s0 < a.B; s0 += n_warps * G) {
    const int64_t s = s0 + grp;
    const bool valid = s < a.B;
    const bool mine = valid && lg < F;                 // lane lg of the group looks after field lg
    const int my_id = mine ? __ldg(a.col + s * F + lg) : 0;
    int id[NF];
#pragma unroll
    for (int f = 0; f < NF; f++) id[f] = __shfl_sync(0xffffffffu, my_id, grp * LPS + (f < LPS ? f : 0));
    float4 e[NF];
#pragma unroll
    for (int f = 0; f < NF; f++) e[f] = (valid && f < F) ? ldg4(V4 + (size_t)id[f] * LPS + lg) : f4_zero();
    const int my_slot = (mine && a.hot.slot) ? __ldg(a.hot.slot + my_id) : -1;
    const float my_bias = (mine && a.bias) ? __ldg(a.bias + my_id) : 0.f;
    const float y = valid ? __ldg(a.labels + s) : 0.f;

    float4 S = f4_zero(), Q = f4_zero();
#pragma unroll
    for (int f = 0; f < NF; f++) {                      // fields in order (FM.py:100,105-106)
      S = f4_add(S, e[f]);
      Q = f4_add(Q, f4_mul(e[f], e[f]));
    }
    const float part = 0.5f * f4_hsum(f4_sub(f4_mul(S, S), Q));
    // bias terms are summed in field order by the group leader to match the generic kernel / oracle order
    float bsum = 0.f;
#pragma unroll
    for (int f = 0; f < NF; f++) {
      const float bf = __shfl_sync(0xffffffffu, my_bias, grp * LPS + (f < LPS ? f : 0));
      if (f < F) bsum += bf;
    }
    const float bil = group_sum<LPS>(part);
    const float out = (bil + bsum) + b0;
    const float diff = y - out;
    const float g = valid ? -diff : 0.f;
    if (valid && lg == 0) {
      loss_acc += 0.5f * diff * diff;
      g0_acc += g;
      if (a.out) a.out[s] = out;
    }
    // ---- backward: gV[x_f] += g*(S - e_f) (one REDG.128 per lane and field); gbias[x_f] += g ----
#pragma unroll
    for (int f = 0; f < NF; f++) {
      const int slot = __shfl_sync(0xffffffffu, my_slot, grp * LPS + (f < LPS ? f : 0));
      if (valid && f < F) {
        float* dst = (slot >= 0) ? a.hot.ghot + ((size_t)rep * a.hot.n_hot + slot) * K : a.gV + (size_t)id[f] * K;
        red_add_v4(dst + 4 * lg, f4_scale(f4_sub(S, e[f]), g));
      }
    }
    if (mine && a.gbias) {
      float* p = a.gbias + my_id;
      if (my_slot >= 0 && a.hot.ghot_bias != nullptr) p = a.hot.ghot_bias + (size_t)rep * a.hot.n_hot + my_slot;
      atomicAdd(p, g);
    }
    if (a.touch_stamp != nullptr) {
      // first toucher of a row in this step claims it; the claims of a warp share one counter atomic
      bool claimed = false;
      if (mine && __ldcv(a.touch_stamp + my_id) != a.stamp) claimed = atomicExch(a.touch_stamp + my_id, a.stamp) != a.stamp;
      const unsigned m = __ballot_sync(0xffffffffu, claimed);
      if (m) {
        const int leader = __ffs(m) - 1;
        int base = 0;
        if (lane == leader) base = atomicAdd(a.touched_count, __popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (claimed) a.touched_rows[base + __popc(m & ((1u << lane) - 1))] = my_id;
      }
    }
  }
  const float bl = block_sum(loss_acc, scratch);
  write_partial(a.loss_partials, bl);
  if (a.gb0 != nullptr) {
    const float bg = block_sum(g0_acc, scratch);
    if (threadIdx.x == 0 && bg != 0.f) atomicAdd(a.gb0, bg);
  }
}

template <int LPS, int NF>
static int launch_fm_fixed(const FmArgs& a, cudaStream_t st) {
  static int occ = 0;
  if (occ == 0) {
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fm_train_fixed_kernel<LPS, NF>, kBlock, 0);
    if (occ < 1) occ = 1;
  }
  const int grid = grid_for(a.B, (kBlock / 32) * (32 / LPS), occ);
  fm_train_fixed_kernel<LPS, NF><<<grid, kBlock, 0, st>>>(a);
  return check_launch("fm_train_fixed_kernel");
}

// Returns HHFM_ERR_UNSUPPORTED when the shape is not covered (the caller then uses the generic kernel).
static int dispatch_fm_fixed(const FmArgs& a, cudaStream_t st) {
  if (a.row_ptr != nullptr || a.val != nullptr || a.interaction != 0) return HHFM_ERR_UNSUPPORTED;
  const int lps = a.K / 4;
  if (a.K != 32 && a.K != 64 && a.K != 128) return HHFM_ERR_UNSUPPORTED;
  if (a.F > 16 || a.F > lps) return HHFM_ERR_UNSUPPORTED;
#define FIXED(L)                                              \
  do {                                                        \
    if (a.F <= 8) return launch_fm_fixed<L, 8>(a, st);        \
    if (a.F <= 12) return launch_fm_fixed<L, 12>(a, st);      \
    return launch_fm_fixed<L, 16>(a, st);                     \
  } while (0)
  if (lps == 8) return launch_fm_fixed<8, 8>(a, st);          // F <= K/4 = 8
  if (lps == 16) FIXED(16);
  FIXED(32);
#undef FIXED
}

// ---------------------------------------------------------------------------------------------------------------
// TMA-staged training kernel for tables that do not fit in L2 (scaled config: M = 10^7, K = 128, 5 GB of rows).
// The register kernel above is bounded by memory latency there (ncu: DRAM 29 %, every warp in long-scoreboard stalls,
// 16 warps/SM x 10 gathers in flight).  Here every warp runs its own NS-deep pipeline in shared memory:
//   iteration t:  (A) LDGSTS the ids of sample t                                     -> id ring
//                 (B) sample t-PD: one bulk copy (cp.async.bulk, UBLKCP) per field row -> row stage, completion on the
//                     stage's mbarrier; LDGSTS of bias[id] / hot_slot[id]              -> per-stage side buffers
//                 (C) sample t-PD-NS+1: wait on its mbarrier, FM forward + loss + backward from shared memory
// so NS*F rows (NS*F*K*4 bytes, 20 KB at F=10, K=128) are in flight per warp with no register cost, and no load of
// the consumer step (C) goes to global memory.  Touched rows are marked with a plain store into the stamp array and
// compacted into the list afterwards (touched_compact_kernel) instead of one returning atomic per row.
constexpr int kStagedWarps = 10;
constexpr int kStagedMaxF = 16;

// shared memory per warp: NS row stages [F][K] floats, then (NS+PD) id slots, NS bias slots, NS hot-slot slots of
// kStagedMaxF words each, then NS mbarriers.
__host__ __device__ inline size_t staged_warp_bytes(int NS, int F, int K) {
  const int PD = NS - 1;
  const size_t b = (size_t)NS * F * K * 4 + (size_t)((NS + PD) + 2 * NS) * kStagedMaxF * 4 + (size_t)NS * 8;
  return (b + 127) / 128 * 128;
}

template <int NS, int NW = kStagedWarps>
__global__ void __launch_bounds__(NW * 32, 1) fm_train_staged_kernel(const FmArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ float scratch[32];
  constexpr int PD = NS - 1;          // id prefetch distance (iterations)
  constexpr int RI = NS + PD;         // id ring slots
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = a.F, K = a.K, kv = K >> 2;
  const uint32_t row_bytes = (uint32_t)K * 4u;
  unsigned char* base = smem_raw + (size_t)warp * staged_warp_bytes(NS, F, K);
  float* rows = reinterpret_cast<float*>(base);                                   // [NS][F][K]
  int* idring = reinterpret_cast<int*>(base + (size_t)NS * F * K * 4);             // [RI][16]
  float* biasbuf = reinterpret_cast<float*>(idring + RI * kStagedMaxF);            // [NS][16]
  int* slotbuf = reinterpret_cast<int*>(biasbuf + NS * kStagedMaxF);               // [NS][16]
  uint64_t* bars = reinterpret_cast<uint64_t*>(slotbuf + NS * kStagedMaxF);        // [NS]
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NS; i++) mbar_init1(bars + i);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncwarp();

  // contiguous range of samples per warp: consecutive iterations read consecutive id records
  const int64_t n_warps = (int64_t)gridDim.x * NW;
  const int64_t warp_g = (int64_t)blockIdx.x * NW + warp;
  const int64_t per = (a.B + n_warps - 1) / n_warps;
  const int64_t s_beg = warp_g * per;
  const int64_t s_end = (s_beg + per < a.B) ? s_beg + per : a.B;
  const int64_t n = s_end > s_beg ? s_end - s_beg : 0;
  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  const int rep = a.hot.slot ? (int)(warp_g % a.hot.n_rep) : 0;
  float loss_acc = 0.f, g0_acc = 0.f;

  for (int64_t t = 0; t < n + PD + NS - 1; t++) {
    // (A) ids of sample t
    if (t < n && lane < F) ldgsts4(idring + (t % RI) * kStagedMaxF + lane, a.col + (s_beg + t) * F + lane);
    // Group t (committed below) = {ids of sample t, bias / hot-slot words of sample t-PD}.  Groups <= t-PD are complete
    // after this wait (the PD-1 most recent committed ones may be pending): the ids of sample t-PD and, since
    // PD == NS-1, the bias / hot-slot words of the sample consumed in this iteration.
    ldgsts_wait<(PD > 0 ? PD - 1 : 0)>();
    __syncwarp();
    // (B) issue the row copies of sample j
    const int64_t j = t - PD;
    if (j >= 0 && j < n) {
      const int st = (int)(j % NS);
      if (lane == 0) mbar_expect(bars + st, row_bytes * (uint32_t)F);
      __syncwarp();
      if (lane < F) {
        const int id = idring[(j % RI) * kStagedMaxF + lane];
        bulk_row(rows + ((size_t)st * F + lane) * K, a.V + (size_t)id * K, row_bytes, bars + st);
        if (a.bias) ldgsts4(biasbuf + st * kStagedMaxF + lane, a.bias + id);
        if (a.hot.slot) ldgsts4(slotbuf + st * kStagedMaxF + lane, a.hot.slot + id);
      }
    }
    ldgsts_commit();
    // (C) consume sample c
    const int64_t c = t - PD - NS + 1;
    if (c >= 0 && c < n) {
      const int st = (int)(c % NS);
      const int64_t s = s_beg + c;
      mbar_wait_parity(bars + st, (uint32_t)((c / NS) & 1));
      const float4* r4 = reinterpret_cast<const float4*>(rows + (size_t)st * F * K);
      const int* ids = idring + (c % RI) * kStagedMaxF;
      float4 S[4], Q[4];
#pragma unroll
      for (int i = 0; i < 4; i++) { S[i] = f4_zero(); Q[i] = f4_zero(); }
      for (int f = 0; f < F; f++) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int cc = lane + 32 * i;
          if (cc < kv) {
            const float4 e = r4[f * kv + cc];
            S[i] = f4_add(S[i], e);
            Q[i] = f4_add(Q[i], f4_mul(e, e));
          }
        }
      }
      float part = 0.f;
#pragma unroll
      for (int i = 0; i < 4; i++) part += 0.5f * f4_hsum(f4_sub(f4_mul(S[i], S[i]), Q[i]));
      float bsum = 0.f;
      if (a.bias)
        for (int f = 0; f < F; f++) bsum += biasbuf[st * kStagedMaxF + f];
      const float out = (warp_sum(part) + bsum) + b0;
      const float diff = __ldg(a.labels + s) - out;
      const float g = -diff;
      if (lane == 0) {
        loss_acc += 0.5f * diff * diff;
        g0_acc += g;
        if (a.out) a.out[s] = out;
      }
      for (int f = 0; f < F; f++) {
        const int id = ids[f];
        const int slot = a.hot.slot ? slotbuf[st * kStagedMaxF + f] : -1;
        float* dst = (slot >= 0) ? a.hot.ghot + ((size_t)rep * a.hot.n_hot + slot) * K : a.gV + (size_t)id * K;
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int cc = lane + 32 * i;
          if (cc < kv) red_add_v4(dst + 4 * cc, f4_scale(f4_sub(S[i], r4[f * kv + cc]), g));
        }
      }
      if (lane < F) {
        const int id = ids[lane];
        if (a.gbias) {
          const int slot = a.hot.slot ? slotbuf[st * kStagedMaxF + lane] : -1;
          float* p = (slot >= 0 && a.hot.ghot_bias != nullptr) ? a.hot.ghot_bias + (size_t)rep * a.hot.n_hot + slot : a.gbias + id;
          atomicAdd(p, g);
        }
        if (a.touch_stamp) a.touch_stamp[id] = a.stamp;       // compacted into the list by touched_compact_kernel
      }
      __syncwarp();     // every lane is done with this stage before the next iteration re-arms it
    }
  }
  ldgsts_wait<0>();
  const float bl = block_sum(loss_acc, scratch);
  write_partial(a.loss_partials, bl);
  if (a.gb0 != nullptr) {
    const float bg = block_sum(g0_acc, scratch);
    if (threadIdx.x == 0 && bg != 0.f) atomicAdd(a.gb0, bg);
  }
}

// rows whose stamp equals `stamp` -> appended to list[*count ...].  Four stamps per thread (one 16-byte load), the hits of a
// CTA round are ranked with a warp ballot + a 8-entry scan in shared memory, ONE counter atomic per CTA and round (the first
// version took one per warp: 3 x 10^5 atomics on one address at M = 10^7, 176 us for a 40 MB read).
__global__ void __launch_bounds__(256) touched_compact_kernel(const int32_t* __restrict__ stamp_arr, int32_t stamp, int64_t M,
                                                              int32_t* __restrict__ list, int32_t* __restrict__ count) {
  __shared__ int warp_cnt[8];
  __shared__ int cta_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n4 = M >> 2;                                    // whole int4 groups; the tail is handled by the last CTA round
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t rounds = ((n4 + 1) + stride - 1) / stride;
  for (int64_t r = 0; r < rounds; r++) {
    const int64_t i = r * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int4 v = make_int4(stamp - 1, stamp - 1, stamp - 1, stamp - 1);
    if (i < n4) {
      v = __ldg(reinterpret_cast<const int4*>(stamp_arr) + i);
    } else if (i == n4) {
      const int64_t b = n4 << 2;
      if (b < M) v.x = __ldg(stamp_arr + b);
      if (b + 1 < M) v.y = __ldg(stamp_arr + b + 1);
      if (b + 2 < M) v.z = __ldg(stamp_arr + b + 2);
    }
    const int h0 = v.x == stamp, h1 = v.y == stamp, h2 = v.z == stamp, h3 = v.w == stamp;
    const int mine = h0 + h1 + h2 + h3;
    int incl = mine;                                            // inclusive scan over the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_cnt[warp] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
#pragma unroll
      for (int w = 0; w < 8; w++) { const int c = warp_cnt[w]; warp_cnt[w] = tot; tot += c; }
      cta_base = tot ? atomicAdd(count, tot) : 0;
    }
    __syncthreads();
    if (mine) {
      int p = cta_base + warp_cnt[warp] + incl - mine;
      const int32_t e = (int32_t)(i << 2);
      if (h0) list[p++] = e;
      if (h1) list[p++] = e + 1;
      if (h2) list[p++] = e + 2;
      if (h3) list[p++] = e + 3;
    }
    __syncthreads();                                            // warp_cnt / cta_base are rewritten by the next round
  }
}

// fallback for a stamp array that is not 16-byte aligned (one counter atomic per warp)
__global__ void __launch_bounds__(256) touched_compact_scalar_kernel(const int32_t* __restrict__ stamp_arr, int32_t stamp, int64_t M,
                                                                     int32_t* __restrict__ list, int32_t* __restrict__ count) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t rounds = (M + stride - 1) / stride;
  for (int64_t r = 0; r < rounds; r++) {
    const int64_t i = r * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool hit = (i < M) && (__ldg(stamp_arr + i) == stamp);
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (m) {
      const int leader = __ffs(m) - 1;
      int basep = 0;
      if (lane == leader) basep = atomicAdd(count, __popc(m));
      basep = __shfl_sync(0xffffffffu, basep, leader);
      if (hit) list[basep + __popc(m & ((1u << lane) - 1))] = (int32_t)i;
    }
  }
}

int launch_touched_compact(const int32_t* stamp_arr, int32_t stamp, int64_t M, int32_t* list, int32_t* count, cudaStream_t st) {
  const bool vec = ((uintptr_t)stamp_arr & 15) == 0;
  int64_t blocks = vec ? (M / 4 + 1 + 255) / 256 : (M + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  if (vec) touched_compact_kernel<<<(int)blocks, 256, 0, st>>>(stamp_arr, stamp, M, list, count);
  else touched_compact_scalar_kernel<<<(int)blocks, 256, 0, st>>>(stamp_arr, stamp, M, list, count);
  return check_launch("touched_compact_kernel");
}

// HHFM_ERR_UNSUPPORTED when the shape is not covered or the table is small enough to live in L2 (the register kernel wins
// there); `M` is needed for the stamp compaction.
static int dispatch_fm_staged(const FmArgs& a, int64_t M, cudaStream_t st) {
  if (a.row_ptr != nullptr || a.val != nullptr || a.interaction != 0) return HHFM_ERR_UNSUPPORTED;
  if (a.F > kStagedMaxF || a.K < 64 || a.K > 512) return HHFM_ERR_UNSUPPORTED;
  const char* env = getenv("HHFM_FM_STAGED");       // 0 = never, 1 = always, unset = by table size
  const int force = env ? (env[0] == '1' ? 1 : 0) : 2;
  if (force == 0) return HHFM_ERR_UNSUPPORTED;
  if (force == 2 && (size_t)M * a.K * 4 < ((size_t)96 << 20)) return HHFM_ERR_UNSUPPORTED;
  const size_t cap = (size_t)224 * 1024;
  // measured at the c5 shape (F = 10, K = 128): 10 warps x 4 stages 5.95 ms per step, 10 x 3 5.91, 11 x 3 5.64, 12 x 3 5.74,
  // 13 x 3 5.81, 14 x 3 5.88, 16 x 2 5.92 -> eleven warps with three stages each when that fits
  int ns = 4, nw = kStagedWarps;
  if (staged_warp_bytes(3, a.F, a.K) * 11 <= cap && staged_warp_bytes(4, a.F, a.K) * kStagedWarps > (size_t)200 * 1024) { ns = 3; nw = 11; }
  const char* ens = getenv("HHFM_FM_STAGES");              // 2..4: pipeline depth (A/B runs)
  if (ens && ens[0] >= '2' && ens[0] <= '4') ns = ens[0] - '0';
  const char* enw = getenv("HHFM_FM_WARPS");               // 10 .. 14 / 16 warps per CTA (A/B runs)
  if (enw) { const int v = atoi(enw); if ((v >= 10 && v <= 14) || v == 16) nw = v; }
  while (ns > 2 && staged_warp_bytes(ns, a.F, a.K) * nw > cap) ns--;
  const size_t smem = staged_warp_bytes(ns, a.F, a.K) * nw;
  if (smem > cap) return HHFM_ERR_UNSUPPORTED;
  const int grid = sm_count();
  if (grid > kPartials) return HHFM_ERR_UNSUPPORTED;
  cudaError_t e = cudaSuccess;
#define HHFM_LAUNCH_STAGED(NS_, NW_)                                                                                              \
  do {                                                                                                                            \
    e = cudaFuncSetAttribute(fm_train_staged_kernel<NS_, NW_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
    if (e == cudaSuccess) fm_train_staged_kernel<NS_, NW_><<<grid, NW_ * 32, smem, st>>>(a);                                      \
  } while (0)
  if (nw == kStagedWarps) {
    if (ns == 4) HHFM_LAUNCH_STAGED(4, kStagedWarps);
    else if (ns == 3) HHFM_LAUNCH_STAGED(3, kStagedWarps);
    else HHFM_LAUNCH_STAGED(2, kStagedWarps);
  } else if (nw == 11) {
    if (ns >= 3) HHFM_LAUNCH_STAGED(3, 11);
    else HHFM_LAUNCH_STAGED(2, 11);
  } else if (nw == 13) {
    if (ns >= 3) HHFM_LAUNCH_STAGED(3, 13);
    else HHFM_LAUNCH_STAGED(2, 13);
  } else if (nw == 12) {
    if (ns >= 3) HHFM_LAUNCH_STAGED(3, 12);
    else HHFM_LAUNCH_STAGED(2, 12);
  } else if (nw == 14) {
    if (ns >= 3) HHFM_LAUNCH_STAGED(3, 14);
    else HHFM_LAUNCH_STAGED(2, 14);
  } else {
    HHFM_LAUNCH_STAGED(2, 16);
  }
#undef HHFM_LAUNCH_STAGED
  if (e != cudaSuccess) {
    set_error("fm_train_staged_kernel: %s", cudaGetErrorString(e));
    return HHFM_ERR_LAUNCH;
  }
  int rc = check_launch("fm_train_staged_kernel");
  if (rc != HHFM_OK) return rc;
  if (a.touch_stamp != nullptr) rc = launch_touched_compact(a.touch_stamp, a.stamp, M, a.touched_rows, a.touched_count, st);
  return rc;
}

template <int LPS, int VPL, int MODE, bool DROP = false>
static int launch_fm(const FmArgs& a, int deterministic, cudaStream_t st) {
  static int occ = 0;
  if (occ == 0) {
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fm_kernel<LPS, VPL, MODE, DROP>, kBlock, 0);
    if (occ < 1) occ = 1;
  }
  FmArgs b = a;
  constexpr int G = 32 / LPS;
  if (deterministic) {
    b.groups_active = 1;
    fm_kernel<LPS, VPL, MODE, DROP><<<1, 32, 0, st>>>(b);
  } else {
    b.groups_active = G;
    const int grid = grid_for(a.B, (kBlock / 32) * G, occ);
    fm_kernel<LPS, VPL, MODE, DROP><<<grid, kBlock, 0, st>>>(b);
  }
  return check_launch("fm_kernel");
}

template <int MODE>
static int dispatch_fm(const FmArgs& a, int deterministic, cudaStream_t st) {
#define CALL(L, V) return launch_fm<L, V, MODE>(a, deterministic, st)
  HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  return HHFM_ERR_UNSUPPORTED;
}

static int dispatch_fm_train_dropout(const FmArgs& a, int deterministic, cudaStream_t st) {
#define CALL(L, V) return launch_fm<L, V, FM_TRAIN, true>(a, deterministic, st)
  HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  return HHFM_ERR_UNSUPPORTED;
}

static int check_common(int64_t B, int64_t F, const void* col, const void* V, int64_t M, int64_t K, int interaction,
                        const void* row_ptr) {
  HHFM_REQUIRE(B >= 0 && M > 0, "fm: bad sizes B=%lld M=%lld", (long long)B, (long long)M);
  HHFM_REQUIRE(col != nullptr && V != nullptr, "fm: col and V must not be NULL");
  HHFM_REQUIRE(K > 0 && K % 4 == 0 && K <= 512, "fm: K=%lld unsupported (need K %% 4 == 0, K <= 512)", (long long)K);
  HHFM_REQUIRE(row_ptr != nullptr || F > 0, "fm: fixed-width batch needs F > 0");
  HHFM_REQUIRE(interaction == 0 || interaction == 1, "fm: interaction must be 0 (FM) or 1 (MF)");
  HHFM_REQUIRE(interaction == 0 || (row_ptr == nullptr && F >= 2), "fm: MF interaction needs fixed width F >= 2");
  HHFM_REQUIRE(((uintptr_t)V & 15) == 0, "fm: V must be 16-byte aligned");
  return HHFM_OK;
}

}  // namespace hhfm

using namespace hhfm;

extern "C" int hhfm_fm_fwd(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B, int64_t F,
                           const float* V, const float* bias, const float* b0, int64_t M, int64_t K,
                           int32_t interaction, float* out, hhfm_stream_t stream) {
  int rc = check_common(B, F, col, V, M, K, interaction, row_ptr);
  if (rc) return rc;
  HHFM_REQUIRE(out != nullptr, "fm_fwd: out is NULL");
  if (B == 0) return HHFM_OK;
  FmArgs a{};
  a.row_ptr = row_ptr; a.col = col; a.val = val; a.B = B; a.F = (int)F; a.V = V; a.bias = bias; a.b0 = b0;
  a.K = (int)K; a.interaction = interaction; a.out = out;
  return dispatch_fm<FM_FWD>(a, 0, (cudaStream_t)stream);
}

extern "C" int hhfm_fm_fwd_bwd_sqloss_dropout(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B,
                                      int64_t F, const float* V, const float* bias, const float* b0, int64_t M,
                                      int64_t K, int32_t interaction, const float* labels, float* out, float* gV,
                                      float* gbias, float* gb0, float* loss_partials, int32_t* touch_stamp,
                                      int32_t stamp, int32_t* touched_rows, int32_t* touched_count,
                                      const int32_t* hot_slot, float* ghot, float* ghot_bias, int32_t n_rep,
                                      int32_t n_hot, int32_t deterministic, float keep, uint64_t drop_seed, hhfm_stream_t stream) {
  int rc = check_common(B, F, col, V, M, K, interaction, row_ptr);
  if (rc) return rc;
  HHFM_REQUIRE(!hot_slot || (ghot && n_rep >= 1 && n_hot >= 1), "fm_fwd_bwd_sqloss: hot_slot needs ghot, n_rep, n_hot");
  HHFM_REQUIRE(labels && gV && loss_partials, "fm_fwd_bwd_sqloss: labels, gV and loss_partials are required");
  HHFM_REQUIRE(B > 0, "fm_fwd_bwd_sqloss: empty batch");
  HHFM_REQUIRE(!touch_stamp || (touched_rows && touched_count), "fm_fwd_bwd_sqloss: touch_stamp needs touched_rows/count");
  HHFM_REQUIRE(((uintptr_t)gV & 15) == 0, "fm: gV must be 16-byte aligned");
  FmArgs a{};
  a.row_ptr = row_ptr; a.col = col; a.val = val; a.B = B; a.F = (int)F; a.V = V; a.bias = bias; a.b0 = b0;
  a.K = (int)K; a.interaction = interaction; a.labels = labels; a.out = out; a.gV = gV; a.gbias = gbias; a.gb0 = gb0;
  a.loss_partials = loss_partials; a.touch_stamp = touch_stamp; a.stamp = stamp; a.touched_rows = touched_rows;
  a.touched_count = touched_count;
  a.hot = HotPlan{hot_slot, ghot, ghot_bias, n_rep, n_hot};
  HHFM_REQUIRE(keep > 0.f && keep <= 1.f, "fm_fwd_bwd_sqloss: dropout keep must be in (0, 1]");
  a.keep = keep;
  a.drop_seed = drop_seed;
  if (keep < 1.f) return dispatch_fm_train_dropout(a, deterministic, (cudaStream_t)stream);
  if (!deterministic) {
    rc = dispatch_fm_staged(a, M, (cudaStream_t)stream);
    if (rc != HHFM_ERR_UNSUPPORTED) return rc;
    rc = dispatch_fm_fixed(a, (cudaStream_t)stream);
    if (rc != HHFM_ERR_UNSUPPORTED) return rc;
  }
  return dispatch_fm<FM_TRAIN>(a, deterministic, (cudaStream_t)stream);
}

extern "C" int hhfm_fm_fwd_bwd_sqloss(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B,
                                      int64_t F, const float* V, const float* bias, const float* b0, int64_t M,
                                      int64_t K, int32_t interaction, const float* labels, float* out, float* gV,
                                      float* gbias, float* gb0, float* loss_partials, int32_t* touch_stamp,
                                      int32_t stamp, int32_t* touched_rows, int32_t* touched_count,
                                      const int32_t* hot_slot, float* ghot, float* ghot_bias, int32_t n_rep,
                                      int32_t n_hot, int32_t deterministic, hhfm_stream_t stream) {
  return hhfm_fm_fwd_bwd_sqloss_dropout(row_ptr, col, val, B, F, V, bias, b0, M, K, interaction, labels, out, gV, gbias, gb0,
                                        loss_partials, touch_stamp, stamp, touched_rows, touched_count, hot_slot, ghot,
                                        ghot_bias, n_rep, n_hot, deterministic, 1.0f, 0ull, stream);
}

extern "C" int hhfm_fm_bwd(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B, int64_t F,
                           const float* V, int64_t M, int64_t K, int32_t interaction, const float* gout, float* gV,
                           float* gbias, float* gb0, int32_t deterministic, hhfm_stream_t stream) {
  int rc = check_common(B, F, col, V, M, K, interaction, row_ptr);
  if (rc) return rc;
  HHFM_REQUIRE(gout && gV, "fm_bwd: gout and gV are required");
  if (B == 0) return HHFM_OK;
  FmArgs a{};
  a.row_ptr = row_ptr; a.col = col; a.val = val; a.B = B; a.F = (int)F; a.V = V; a.K = (int)K;
  a.interaction = interaction; a.gout = gout; a.gV = gV; a.gbias = gbias; a.gb0 = gb0;
  return dispatch_fm<FM_BWD>(a, deterministic, (cudaStream_t)stream);
}
