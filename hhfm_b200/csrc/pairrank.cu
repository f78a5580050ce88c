// K3: HHFM (OurModel7.py:105-184) and BPR (BPR.py:76-88) pairwise ranking with max-negative, fused:
// group pooling -> hybrid feature -> positive / negative dots -> reduce_max -> -log(sigmoid) -> gradients ->
// sort-free scatter (REDG.E.ADD.F32x4).  Same lane mapping as fm.cu: LPS = K/4 lanes own one sample.
//
// Record (int32, `stride` ints, 16-byte aligned): [user, item+, ctx.., time.., neg.., pad].
#include <stdlib.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "staged.cuh"

namespace hhfm {

struct PrArgs {
  const int32_t* idx;
  int64_t B;
  int stride;
  int n_ctx, n_time, n_neg;
  int pc, pt, pf;
  const float* V;
  int K;
  float* pos_out;
  float* neg_out;
  const float* dpos;
  const float* dneg;
  float* gV;
  float* loss_partials;
  int32_t* touch_stamp;
  int32_t stamp;
  int32_t* touched_rows;
  int32_t* touched_count;
  int groups_active;
  HotPlan hot;
};

enum { PR_FWD = 0, PR_TRAIN = 1, PR_BWD = 2 };

// Pool n rows V[ids[0..n)] element-wise (OurModel7.py:124/141 Pooling1C/Pooling1T over axis=1).
// MAX keeps the per-element tie count for the reduce_max gradient.  Rows are combined in id order.
template <int LPS, int VPL, bool ANYMAX>
__device__ __forceinline__ void pool_rows(const float* __restrict__ V, const int32_t* __restrict__ ids, int n, int mode,
                                          int K, int lg, Frag<LPS, VPL>& out, Frag<LPS, VPL>& cnt) {
  using F4 = Frag<LPS, VPL>;
  frag_zero(out);
  if (ANYMAX) frag_zero(cnt);
  for (int j = 0; j < n; j += 4) {
    int id[4];
    F4 e[4];
#pragma unroll
    for (int u = 0; u < 4; u++) id[u] = (j + u < n) ? __ldg(ids + j + u) : -1;
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (id[u] >= 0) frag_load(e[u], V, id[u], K, lg);
#pragma unroll
    for (int u = 0; u < 4; u++) {
      if (id[u] < 0) continue;
      if (ANYMAX && mode == HHFM_POOL_MAX) {
        const bool first = (j + u) == 0;
#pragma unroll
        for (int i = 0; i < VPL; i++) {
          float* o = reinterpret_cast<float*>(&out.v[i]);
          float* c = reinterpret_cast<float*>(&cnt.v[i]);
          const float* x = reinterpret_cast<const float*>(&e[u].v[i]);
#pragma unroll
          for (int q = 0; q < 4; q++) {
            if (first || x[q] > o[q]) { o[q] = x[q]; c[q] = 1.f; }
            else if (x[q] == o[q]) c[q] += 1.f;
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < VPL; i++) out.v[i] = f4_add(out.v[i], e[u].v[i]);
      }
    }
  }
  if (mode == HHFM_POOL_MEAN) {
    const float fn = (float)n;
#pragma unroll
    for (int i = 0; i < VPL; i++)
      out.v[i] = make_float4(out.v[i].x / fn, out.v[i].y / fn, out.v[i].z / fn, out.v[i].w / fn);
  }
}

// Scatter the gradient d of a pooled vector back to its n member rows.
template <int LPS, int VPL, bool ANYMAX>
__device__ __forceinline__ void pool_rows_bwd(const PrArgs& a, int rep, const int32_t* __restrict__ ids, int n, int mode, int lg,
                                              const Frag<LPS, VPL>& pooled, const Frag<LPS, VPL>& cnt,
                                              const Frag<LPS, VPL>& d) {
  using F4 = Frag<LPS, VPL>;
  const int K = a.K;
  F4 dm = d;
  if (mode == HHFM_POOL_MEAN) {
    const float fn = (float)n;
#pragma unroll
    for (int i = 0; i < VPL; i++) dm.v[i] = make_float4(d.v[i].x / fn, d.v[i].y / fn, d.v[i].z / fn, d.v[i].w / fn);
  }
  for (int j = 0; j < n; j++) {
    const int id = __ldg(ids + j);
    if (ANYMAX && mode == HHFM_POOL_MAX) {
      F4 e, r;
      frag_load(e, a.V, id, K, lg);
#pragma unroll
      for (int i = 0; i < VPL; i++) {
        const float* x = reinterpret_cast<const float*>(&e.v[i]);
        const float* o = reinterpret_cast<const float*>(&pooled.v[i]);
        const float* c = reinterpret_cast<const float*>(&cnt.v[i]);
        const float* dd = reinterpret_cast<const float*>(&d.v[i]);
        float* rr = reinterpret_cast<float*>(&r.v[i]);
#pragma unroll
        for (int q = 0; q < 4; q++) rr[q] = (x[q] == o[q]) ? (1.f / c[q]) * dd[q] : 0.f;
      }
      scatter_row<LPS, VPL>(a.gV, a.hot, rep, id, K, lg, r);
    } else {
      scatter_row<LPS, VPL>(a.gV, a.hot, rep, id, K, lg, dm);
    }
    if (lg == 0) touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, id);
  }
}

template <int LPS, int VPL, int MODE, bool ANYMAX>
__global__ void __launch_bounds__(kBlock) pairrank_kernel(const PrArgs a) {
  __shared__ float scratch[32];
  using F4 = Frag<LPS, VPL>;
  const int lane = threadIdx.x & 31, lg = lane % LPS, grp = lane / LPS;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int ga = a.groups_active;
  const int K = a.K;
  const int num = 1 + (a.n_ctx > 0) + (a.n_time > 0);   // OurModel7.py:89,94 self.num
  float loss_acc = 0.f;
  const int rep = a.hot.slot ? (int)((warp_g * (32 / LPS) + grp) % a.hot.n_rep) : 0;

  for (int64_t s0 = warp_g * ga; s0 < a.B; s0 += n_warps * ga) {
    const int64_t s = s0 + grp;
    const bool valid = (grp < ga) && (s < a.B);
    const int64_t sc = valid ? s : (a.B - 1);   // padding groups recompute the last sample, never write
    const int32_t* rec = a.idx + sc * a.stride;
    const int uid = __ldg(rec + 0), pid = __ldg(rec + 1);
    const int32_t* ctx = rec + 2;
    const int32_t* tim = ctx + a.n_ctx;
    const int32_t* neg = tim + a.n_time;

    // ---- forward: hybrid feature (OurModel7.py:105-168) ----
    F4 eu, vp, C, cC, T, cT, hyb, cF;
    frag_load(eu, a.V, uid, K, lg);
    frag_load(vp, a.V, pid, K, lg);
    frag_zero(C); frag_zero(T);
    if (ANYMAX) { frag_zero(cC); frag_zero(cT); frag_zero(cF); }
    if (a.n_ctx > 0) pool_rows<LPS, VPL, ANYMAX>(a.V, ctx, a.n_ctx, a.pc, K, lg, C, cC);
    if (a.n_time > 0) pool_rows<LPS, VPL, ANYMAX>(a.V, tim, a.n_time, a.pt, K, lg, T, cT);
    if (num == 1) {
      hyb = eu;
    } else if (ANYMAX && a.pf == HHFM_POOL_MAX) {
#pragma unroll
      for (int i = 0; i < VPL; i++) {
        const float* xu = reinterpret_cast<const float*>(&eu.v[i]);
        const float* xc = reinterpret_cast<const float*>(&C.v[i]);
        const float* xt = reinterpret_cast<const float*>(&T.v[i]);
        float* o = reinterpret_cast<float*>(&hyb.v[i]);
        float* c = reinterpret_cast<float*>(&cF.v[i]);
#pragma unroll
        for (int q = 0; q < 4; q++) {
          float m = xu[q], n_ = 1.f;
          if (a.n_ctx > 0) { if (xc[q] > m) { m = xc[q]; n_ = 1.f; } else if (xc[q] == m) n_ += 1.f; }
          if (a.n_time > 0) { if (xt[q] > m) { m = xt[q]; n_ = 1.f; } else if (xt[q] == m) n_ += 1.f; }
          o[q] = m; c[q] = n_;
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < VPL; i++) {
        float4 h = eu.v[i];
        if (a.n_ctx > 0) h = f4_add(h, C.v[i]);
        if (a.n_time > 0) h = f4_add(h, T.v[i]);
        if (a.pf == HHFM_POOL_MEAN) { const float fn = (float)num; h = make_float4(h.x / fn, h.y / fn, h.z / fn, h.w / fn); }
        hyb.v[i] = h;
      }
    }

    // ---- scores: OurModel7.py:171-174 / BPR.py:79-81 ----
    const float pos = group_sum<LPS>(frag_dot(hyb, vp));
    float m = -INFINITY;
    unsigned long long tie = 0ull;    // bit j set <=> neg_j equals the running max
    for (int j = 0; j < a.n_neg; j += 4) {
      int id[4];
      F4 e[4];
      float p[4];
#pragma unroll
      for (int u = 0; u < 4; u++) id[u] = (j + u < a.n_neg) ? __ldg(neg + j + u) : -1;
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (id[u] >= 0) frag_load(e[u], a.V, id[u], K, lg);
#pragma unroll
      for (int u = 0; u < 4; u++) p[u] = (id[u] >= 0) ? frag_dot(hyb, e[u]) : 0.f;
#pragma unroll
      for (int u = 0; u < 4; u++) p[u] = group_sum<LPS>(p[u]);
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if (id[u] < 0) continue;
        if (p[u] > m) { m = p[u]; tie = 1ull << (j + u); }
        else if (p[u] == m) tie |= 1ull << (j + u);
        if (a.neg_out && valid && lg == 0) a.neg_out[s * a.n_neg + j + u] = p[u];
      }
    }
    if (a.pos_out && valid && lg == 0) a.pos_out[s] = pos;

    if (MODE != PR_FWD && valid) {
      // ---- loss and d loss / d scores ----
      float gp = 0.f, gn = 0.f;   // d/dpos, d/d(each tied max negative)
      if (MODE == PR_TRAIN) {
        const float x = pos - m;
        const float sg = 1.f / (1.f + expf(-x));            // tf.sigmoid
        if (lg == 0) loss_acc += -logf(sg);                  // OurModel7.py:178
        gp = sg - 1.f;                                       // d(-log sigmoid(x))/dx
        gn = -gp / (float)__popcll(tie);                     // reduce_max grad split among ties
      } else {
        gp = __ldg(a.dpos + s);
      }
      // d hyb = gp*v+ + sum_j gn_j*v_j ;  gV[item+] += gp*hyb ; gV[neg_j] += gn_j*hyb
      F4 dh, t;
#pragma unroll
      for (int i = 0; i < VPL; i++) { dh.v[i] = f4_scale(vp.v[i], gp); t.v[i] = f4_scale(hyb.v[i], gp); }
      scatter_row<LPS, VPL>(a.gV, a.hot, rep, pid, K, lg, t);
      if (lg == 0) touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, pid);
      if (MODE == PR_TRAIN) {
        unsigned long long w = tie;
        while (w) {
          const int j = __ffsll((long long)w) - 1;
          w &= w - 1;
          const int id = __ldg(neg + j);
          F4 e;
          frag_load(e, a.V, id, K, lg);
#pragma unroll
          for (int i = 0; i < VPL; i++) { dh.v[i] = f4_fma(e.v[i], gn, dh.v[i]); t.v[i] = f4_scale(hyb.v[i], gn); }
          scatter_row<LPS, VPL>(a.gV, a.hot, rep, id, K, lg, t);
          if (lg == 0) touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, id);
        }
      } else if (a.dneg != nullptr) {
        for (int j = 0; j < a.n_neg; j++) {
          const float c = __ldg(a.dneg + s * a.n_neg + j);
          const int id = __ldg(neg + j);
          F4 e;
          frag_load(e, a.V, id, K, lg);
#pragma unroll
          for (int i = 0; i < VPL; i++) { dh.v[i] = f4_fma(e.v[i], c, dh.v[i]); t.v[i] = f4_scale(hyb.v[i], c); }
          scatter_row<LPS, VPL>(a.gV, a.hot, rep, id, K, lg, t);
          if (lg == 0) touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, id);
        }
      }
      // ---- back through Pooling1F over stack[user, C, T] ----
      F4 du = dh, dC = dh, dT = dh;
      if (num > 1) {
        if (ANYMAX && a.pf == HHFM_POOL_MAX) {
#pragma unroll
          for (int i = 0; i < VPL; i++) {
            const float* h = reinterpret_cast<const float*>(&hyb.v[i]);
            const float* c = reinterpret_cast<const float*>(&cF.v[i]);
            const float* d = reinterpret_cast<const float*>(&dh.v[i]);
            const float* xu = reinterpret_cast<const float*>(&eu.v[i]);
            const float* xc = reinterpret_cast<const float*>(&C.v[i]);
            const float* xt = reinterpret_cast<const float*>(&T.v[i]);
            float* ou = reinterpret_cast<float*>(&du.v[i]);
            float* oc = reinterpret_cast<float*>(&dC.v[i]);
            float* ot = reinterpret_cast<float*>(&dT.v[i]);
#pragma unroll
            for (int q = 0; q < 4; q++) {
              const float share = (1.f / c[q]) * d[q];
              ou[q] = (xu[q] == h[q]) ? share : 0.f;
              oc[q] = (xc[q] == h[q]) ? share : 0.f;
              ot[q] = (xt[q] == h[q]) ? share : 0.f;
            }
          }
        } else if (a.pf == HHFM_POOL_MEAN) {
          const float fn = (float)num;
#pragma unroll
          for (int i = 0; i < VPL; i++) {
            du.v[i] = make_float4(dh.v[i].x / fn, dh.v[i].y / fn, dh.v[i].z / fn, dh.v[i].w / fn);
            dC.v[i] = du.v[i];
            dT.v[i] = du.v[i];
          }
        }
      }
      scatter_row<LPS, VPL>(a.gV, a.hot, rep, uid, K, lg, du);
      if (lg == 0) touch_row(a.touch_stamp, a.stamp, a.touched_rows, a.touched_count, uid);
      if (a.n_ctx > 0) pool_rows_bwd<LPS, VPL, ANYMAX>(a, rep, ctx, a.n_ctx, a.pc, lg, C, cC, dC);
      if (a.n_time > 0) pool_rows_bwd<LPS, VPL, ANYMAX>(a, rep, tim, a.n_time, a.pt, lg, T, cT, dT);
    }
  }

  if (MODE == PR_TRAIN) {
    const float bl = block_sum(loss_acc, scratch);
    write_partial(a.loss_partials, bl);
  }
}

// ---------------------------------------------------------------------------------------------------
// Fast path of the fused training pass for the reference's default configuration: every Pooling1* is
// tf.reduce_sum (OurModel7.py:14-19), so context and time rows are interchangeable (all are summed into the
// hybrid feature and all receive d_hyb), K == 4*LPS, and the group widths are compile-time constants:
// NP = n_ctx + n_time pooled rows, NNEG negatives.  Everything is unrolled: the record is read with int4 loads,
// all NP + NNEG + 2 row gathers are independent LDG.128s, no bound or mode tests remain in the loop.
// The hybrid feature is summed in record order, ((u + c0) + c1) + ..., where the generic kernel pools the group first,
// u + (c0 + c1 + ...): the two differ in the last bit, both are within the 1e-5 parity bar.
// (~3x fewer instructions per sample; see profiles/.)
//
// Pooled context groups (NS < NP, hhfm_pool_groups_attach): the NP pooled columns collapse into NS pooled rows.  Columns
// of a group are replaced by one row of the group table S_g, indexed by the mixed-radix combination of their values
// (pool_groups_presum_kernel sums the member rows into S_g before this kernel), and d_hyb goes to one row of G_g
// (pool_groups_expand_kernel hands it back to the member rows afterwards).  An ungrouped column is a slot of its own that
// reads V directly.  hyb = (u + slot_0) + slot_1 + ..., where a group slot already holds its members' sum.  A sample
// whose member id lies outside the planned range pools and scatters that group's member rows one by one (same order as
// the pre-sum, so the pooled value is the same).
// ---------------------------------------------------------------------------------------------------
constexpr int kPgMaxCols = 16;    // pooled columns (context + time) a plan describes
constexpr int kPgMaxSlots = 4;    // pooled rows per sample after grouping

struct PoolGroups {
  int slot_of[kPgMaxCols];        // pooled column -> slot
  int lo[kPgMaxCols];             // grouped column: first id of its range; ungrouped: 0
  unsigned card[kPgMaxCols];      // grouped column: ids in the range; ungrouped: 0xffffffff (every id qualifies)
  int mult[kPgMaxCols];           // grouped column: mixed-radix weight of its digit; ungrouped: 1
  const float* T[kPgMaxSlots];    // slot table: S_g (group) or V (ungrouped column)
  float* G[kPgMaxSlots];          // group gradient table G_g, nullptr for an ungrouped column
};

template <int LPS, int NP, int NNEG, int NS = NP>
__global__ void __launch_bounds__(kBlock, 2) pairrank_sum_train_kernel(const PrArgs a, const PoolGroups pg) {
  static_assert(NS <= NP, "grouping never adds pooled rows");
  constexpr bool GROUPED = NS < NP;
  __shared__ float scratch[32];
  constexpr int W = 2 + NS + NNEG;                     // gathered rows
  constexpr int W4 = (2 + NP + NNEG + 3) / 4;          // int4 chunks of the record
  const int lane = threadIdx.x & 31, lg = lane % LPS, grp = lane / LPS;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  constexpr int G = 32 / LPS;
  const float4* __restrict__ Vp = reinterpret_cast<const float4*>(a.V) + lg;
  float* __restrict__ Gp = a.gV + 4 * lg;
  const int rep = a.hot.slot ? (int)((warp_g * G + grp) % a.hot.n_rep) : 0;
  float* __restrict__ Hp = a.hot.slot ? a.hot.ghot + (size_t)rep * a.hot.n_hot * (4 * LPS) + 4 * lg : nullptr;
  float loss_acc = 0.f;

  auto scatter = [&](int row, float4 v) {
    float* p = Gp + (size_t)row * (4 * LPS);
    if (Hp != nullptr) {
      const int s = __ldg(a.hot.slot + row);
      if (s >= 0) p = Hp + (size_t)s * (4 * LPS);
    }
    red_add_v4(p, v);
  };

  for (int64_t s0 = warp_g * G; s0 < a.B; s0 += n_warps * G) {
    const int64_t s = s0 + grp;
    const bool valid = s < a.B;
    const int64_t sc = valid ? s : (a.B - 1);
    int idx[W4 * 4];
    const int4* r4 = reinterpret_cast<const int4*>(a.idx + sc * a.stride);
#pragma unroll
    for (int i = 0; i < W4; i++) {
      const int4 t = __ldg(r4 + i);
      idx[4 * i] = t.x; idx[4 * i + 1] = t.y; idx[4 * i + 2] = t.z; idx[4 * i + 3] = t.w;
    }
    float4 e[W];
    int key[NS > 0 ? NS : 1];       // GROUPED: row of each slot's table
    unsigned miss = 0u;             // GROUPED: bit s <=> a member id of slot s lies outside the planned range
    if constexpr (!GROUPED) {
#pragma unroll
      for (int i = 0; i < W; i++) e[i] = __ldg(Vp + (size_t)idx[i] * LPS);
    } else {
#pragma unroll
      for (int q = 0; q < NS; q++) key[q] = 0;
#pragma unroll
      for (int c = 0; c < NP; c++) {              // selects, not a store through slot_of[c]: key stays in registers
        const int d = idx[2 + c] - pg.lo[c], s = pg.slot_of[c], dm = d * pg.mult[c];
        if ((unsigned)d >= pg.card[c]) miss |= 1u << s;
#pragma unroll
        for (int q = 0; q < NS; q++) key[q] += (s == q) ? dm : 0;
      }
      e[0] = __ldg(Vp + (size_t)idx[0] * LPS);
      e[1] = __ldg(Vp + (size_t)idx[1] * LPS);
#pragma unroll
      for (int q = 0; q < NS; q++)
        e[2 + q] = ((miss >> q) & 1u) ? f4_zero()
                                       : __ldg(reinterpret_cast<const float4*>(pg.T[q]) + lg + (size_t)key[q] * LPS);
#pragma unroll
      for (int j = 0; j < NNEG; j++) e[2 + NS + j] = __ldg(Vp + (size_t)idx[2 + NP + j] * LPS);
      if (miss) {                   // fallback: pool the members of the missed slots row by row, in record order
        const int32_t* rec = a.idx + sc * a.stride + 2;
        for (int c = 0; c < NP; c++) {
          const int q = pg.slot_of[c];
          if ((miss >> q) & 1u) {
            const float4 v = __ldg(Vp + (size_t)__ldg(rec + c) * LPS);
#pragma unroll
            for (int qq = 0; qq < NS; qq++)
              if (qq == q) e[2 + qq] = f4_add(e[2 + qq], v);
          }
        }
      }
    }

    float4 hyb = e[0];                                   // user, then ctx.., time.. (or their slots) in record order
#pragma unroll
    for (int i = 0; i < NS; i++) hyb = f4_add(hyb, e[2 + i]);
    float p[1 + NNEG];
    p[0] = f4_dot(hyb, e[1]);
#pragma unroll
    for (int j = 0; j < NNEG; j++) p[1 + j] = f4_dot(hyb, e[2 + NS + j]);
#pragma unroll
    for (int j = 0; j <= NNEG; j++) p[j] = group_sum<LPS>(p[j]);

    // KEEP: the first negative that reaches the max stays in registers (row and id), so the backward pass does not load it
    // again -- one dependent L2 round trip less per sample.  It costs registers: with NP > 0 the kernel stays within the 128
    // of two CTAs per SM (at most 128 in -Xptxas -v), but without context (NP = 0, BPR) it would go from about 80 registers
    // (three CTAs per SM) to about 118 (two), and the lost residency costs more than the load (on a B200, models.bpr_c4:
    // 0.697 -> 0.870 ms per step with KEEP), so NP = 0 loads the row again.
    constexpr bool KEEP = NP > 0;
    float m = p[1];
    unsigned tie = 1u;
    float4 vmax = e[2 + NS];
    int idmax = idx[2 + NP];
#pragma unroll
    for (int j = 1; j < NNEG; j++) {
      if (p[1 + j] > m) {
        m = p[1 + j];
        tie = 1u << j;
        if (KEEP) { vmax = e[2 + NS + j]; idmax = idx[2 + NP + j]; }
      } else if (p[1 + j] == m) {
        tie |= 1u << j;
      }
    }
    if (valid) {
      const float x = p[0] - m;
      const float sg = 1.f / (1.f + expf(-x));
      if (lg == 0) loss_acc += -logf(sg);
      const float gp = sg - 1.f;
      const float gn = -gp / (float)__popc(tie);
      float4 dh = f4_scale(e[1], gp);
      scatter(idx[1], f4_scale(hyb, gp));
      const float4 tn = f4_scale(hyb, gn);
      unsigned w = tie;
      if (KEEP) {                           // further tied negatives (rare) are loaded again, in the same order
        dh = f4_fma(vmax, gn, dh);
        scatter(idmax, tn);
        w &= w - 1u;
      }
      while (w) {
        const int j = __ffs((int)w) - 1;
        w &= w - 1;
        const int id = __ldg(a.idx + sc * a.stride + 2 + NP + j);
        const float4 v = __ldg(Vp + (size_t)id * LPS);
        dh = f4_fma(v, gn, dh);
        scatter(id, tn);
      }
      scatter(idx[0], dh);
      if constexpr (!GROUPED) {
#pragma unroll
        for (int i = 0; i < NP; i++) scatter(idx[2 + i], dh);
      } else {
#pragma unroll
        for (int q = 0; q < NS; q++) {
          if (pg.G[q] == nullptr) scatter(key[q], dh);                          // ungrouped column: key is the row id
          else if (!((miss >> q) & 1u)) red_add_v4(pg.G[q] + (size_t)key[q] * (4 * LPS) + 4 * lg, dh);
        }
        if (miss) {
          const int32_t* rec = a.idx + sc * a.stride + 2;
          for (int c = 0; c < NP; c++)
            if ((miss >> pg.slot_of[c]) & 1u) scatter(__ldg(rec + c), dh);
        }
      }
    }
  }
  const float bl = block_sum(loss_acc, scratch);
  write_partial(a.loss_partials, bl);
}

template <int LPS, int NP, int NNEG, int NS = NP>
static int launch_pr_fast(const PrArgs& a, cudaStream_t st, const PoolGroups& pg = PoolGroups{}) {
  static int occ = 0;
  if (occ == 0) {
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pairrank_sum_train_kernel<LPS, NP, NNEG, NS>, kBlock, 0);
    if (occ < 1) occ = 1;
  }
  constexpr int G = 32 / LPS;
  const int grid = grid_for(a.B, (kBlock / 32) * G, occ);
  pairrank_sum_train_kernel<LPS, NP, NNEG, NS><<<grid, kBlock, 0, st>>>(a, pg);
  return check_launch("pairrank_sum_train_kernel");
}

// returns 1 if the fast path does not cover this configuration
template <int LPS>
static int dispatch_pr_fast_np(const PrArgs& a, cudaStream_t st, int* rc) {
  const int np = a.n_ctx + a.n_time;
  if (a.n_neg != 10) return 1;
  switch (np) {
    case 0: *rc = launch_pr_fast<LPS, 0, 10>(a, st); return 0;
    case 3: *rc = launch_pr_fast<LPS, 3, 10>(a, st); return 0;
    case 8: *rc = launch_pr_fast<LPS, 8, 10>(a, st); return 0;
    case 10: *rc = launch_pr_fast<LPS, 10, 10>(a, st); return 0;
    default: return 1;
  }
}

static int dispatch_pr_fast(const PrArgs& a, cudaStream_t st, int* rc) {
  const bool all_sum = (a.n_ctx == 0 || a.pc == HHFM_POOL_SUM) && (a.n_time == 0 || a.pt == HHFM_POOL_SUM) &&
                       ((a.n_ctx == 0 && a.n_time == 0) || a.pf == HHFM_POOL_SUM);
  if (!all_sum || a.touch_stamp || a.pos_out || a.neg_out) return 1;
  if ((int64_t)a.n_ctx + a.n_time + 2 + a.n_neg > a.stride) return 1;
  switch (a.K) {
    case 32: return dispatch_pr_fast_np<8>(a, st, rc);
    case 64: return dispatch_pr_fast_np<16>(a, st, rc);
    case 128: return dispatch_pr_fast_np<32>(a, st, rc);
    default: return 1;
  }
}

// ---------------------------------------------------------------------------------------------------
// Pooled context groups (include/hhfm_sm100.h hhfm_pool_groups_attach).  A plan is registered under the table pointer V
// and owns its group tables: S (pooled member rows) and G (group gradients, zero between calls), both [rows, K], the
// groups one after another.  One call of the training pass with a matching plan runs
//   pool_groups_presum_kernel  S_g[k] = V[lo_0 + d_0(k)] + V[lo_1 + d_1(k)] + ...   (members in record order)
//   pairrank_sum_train_kernel<LPS, NP, NNEG, NS>
//   pool_groups_expand_kernel  gV[lo_c + d] += sum of G_g[k] over the combinations k with digit d_c(k) == d, fixed order
//   memset(G, 0)
// Nothing else writes a member row of gV during the call (the planner keeps member rows out of the hot-row plan; fallback
// samples reduce into it before the expansion starts, on the same stream), so the expansion adds with a plain
// read-modify-write, and the ranges of grouped columns are disjoint, so no two CTAs of it share a row.
// ---------------------------------------------------------------------------------------------------
struct PgDesc {
  int n_groups;
  int n_mem[kPgMaxSlots];                   // member columns of group g, in record order
  int mem_lo[kPgMaxSlots][kPgMaxCols];
  int mem_card[kPgMaxSlots][kPgMaxCols];
  int64_t row0[kPgMaxSlots + 1];            // first row of group g in S / G; row0[n_groups] = all rows
  int64_t mrow0[kPgMaxSlots + 1];           // first member row of group g in the expansion grid
};

__global__ void __launch_bounds__(kBlock) pool_groups_presum_kernel(const float* __restrict__ V, int K, float* __restrict__ S,
                                                                    const PgDesc d) {
  const int kv = K >> 2;
  const int n = (int)d.row0[d.n_groups] * kv;   // 32-bit index math: at most 2^24 combinations x 32 float4 columns
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int row = i / kv;
    const int j = i - row * kv;
    int g = 0;
    while (g + 1 < d.n_groups && row >= d.row0[g + 1]) g++;
    unsigned k = (unsigned)(row - d.row0[g]);
    float4 acc = f4_zero();
    for (int m = 0; m < d.n_mem[g]; m++) {
      const unsigned c = (unsigned)d.mem_card[g][m], q = k / c;
      const int digit = (int)(k - q * c);
      k = q;
      const float4 v = __ldg(reinterpret_cast<const float4*>(V + (size_t)(d.mem_lo[g][m] + digit) * K) + j);
      acc = (m == 0) ? v : f4_add(acc, v);
    }
    reinterpret_cast<float4*>(S + (size_t)row * K)[j] = acc;
  }
}

// One CTA per member row; thread (lane t % kv, chunk t / kv) sums the float4 column of every combination of its chunk,
// then the chunks are added by a fixed shared-memory tree.
constexpr int kPgExpandThreads = 1024;

__global__ void __launch_bounds__(kPgExpandThreads) pool_groups_expand_kernel(const float* __restrict__ G, int K,
                                                                              float* __restrict__ gV, const PgDesc d) {
  __shared__ float4 part[kPgExpandThreads];
  const int kv = K >> 2;
  const int nchunk = kPgExpandThreads / kv;
  const int j = threadIdx.x % kv, chunk = threadIdx.x / kv;
  const int64_t r = blockIdx.x;
  int g = 0;
  while (g + 1 < d.n_groups && r >= d.mrow0[g + 1]) g++;
  int rem = (int)(r - d.mrow0[g]);          // 32-bit index math: a plan has at most 2^24 combinations
  int m = 0;
  unsigned inner = 1;                       // mixed-radix weight of member m
  while (rem >= d.mem_card[g][m]) { rem -= d.mem_card[g][m]; inner *= (unsigned)d.mem_card[g][m]; m++; }
  const unsigned digit = (unsigned)rem;
  const unsigned span = inner * (unsigned)d.mem_card[g][m];
  const unsigned n = (unsigned)(d.row0[g + 1] - d.row0[g]) / (unsigned)d.mem_card[g][m];   // combinations holding this row
  const float4* Gg = reinterpret_cast<const float4*>(G + (size_t)d.row0[g] * K) + j;
  constexpr int U = 8;
  float4 acc[U];
#pragma unroll
  for (int u = 0; u < U; u++) acc[u] = f4_zero();
  unsigned t = chunk;
  for (; t + (U - 1) * nchunk < n; t += U * nchunk) {
    float4 v[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const unsigned tt = t + u * nchunk, hi = tt / inner;
      v[u] = __ldcg(Gg + (size_t)(tt - hi * inner + digit * inner + hi * span) * kv);
    }
#pragma unroll
    for (int u = 0; u < U; u++) acc[u] = f4_add(acc[u], v[u]);
  }
  for (; t < n; t += nchunk) {
    const unsigned hi = t / inner;
    acc[0] = f4_add(acc[0], __ldcg(Gg + (size_t)(t - hi * inner + digit * inner + hi * span) * kv));
  }
#pragma unroll
  for (int h = U / 2; h > 0; h >>= 1)
#pragma unroll
    for (int u = 0; u < h; u++) acc[u] = f4_add(acc[u], acc[u + h]);
  part[threadIdx.x] = acc[0];
  __syncthreads();
  for (int h = nchunk / 2; h > 0; h >>= 1) {
    if (chunk < h) part[threadIdx.x] = f4_add(part[threadIdx.x], part[threadIdx.x + h * kv]);
    __syncthreads();
  }
  if (chunk == 0) {
    int lo = d.mem_lo[g][m];
    float4* dst = reinterpret_cast<float4*>(gV + (size_t)(lo + digit) * K) + j;
    *dst = f4_add(*dst, part[j]);
  }
}

struct PgPlan {
  const float* V;
  int64_t M;
  int K, n_pool, stride, device;
  int64_t handle;
  int n_slots;
  PoolGroups pg;                            // kernel view of the training pass
  PgDesc desc;                              // pre-sum / expansion view
  float* S;
  float* G;
};

static std::mutex g_pg_mu;
static std::vector<PgPlan*> g_pg_plans;
static int64_t g_pg_next = 1;

static void pg_free(PgPlan* p) {
  cudaFree(p->S);
  cudaFree(p->G);
  delete p;
}

// HHFM_POOL_GROUPS=0 forces the ungrouped kernel (A/B measurements).
static bool pool_groups_enabled() {
  const char* e = getenv("HHFM_POOL_GROUPS");
  return !(e && e[0] == '0');
}

template <int LPS, int NP>
static int launch_pr_grouped_ns(const PrArgs& a, const PgPlan& p, cudaStream_t st, int* rc) {
  switch (p.n_slots) {
    case 1: *rc = launch_pr_fast<LPS, NP, 10, 1>(a, st, p.pg); return 0;
    case 2: *rc = launch_pr_fast<LPS, NP, 10, 2>(a, st, p.pg); return 0;
    case 3: if constexpr (NP > 3) { *rc = launch_pr_fast<LPS, NP, 10, 3>(a, st, p.pg); return 0; } else return 1;
    case 4: if constexpr (NP > 4) { *rc = launch_pr_fast<LPS, NP, 10, 4>(a, st, p.pg); return 0; } else return 1;
    default: return 1;
  }
}

template <int LPS>
static int launch_pr_grouped_np(const PrArgs& a, const PgPlan& p, cudaStream_t st, int* rc) {
  switch (a.n_ctx + a.n_time) {
    case 3: return launch_pr_grouped_ns<LPS, 3>(a, p, st, rc);
    case 8: return launch_pr_grouped_ns<LPS, 8>(a, p, st, rc);
    case 10: return launch_pr_grouped_ns<LPS, 10>(a, p, st, rc);
    default: return 1;
  }
}

// returns 1 if no plan applies (the caller then runs the ungrouped kernels)
static int dispatch_pr_grouped(const PrArgs& a, int64_t M, cudaStream_t st, int* rc) {
  if (!pool_groups_enabled()) return 1;
  const bool all_sum = (a.n_ctx == 0 || a.pc == HHFM_POOL_SUM) && (a.n_time == 0 || a.pt == HHFM_POOL_SUM) &&
                       ((a.n_ctx == 0 && a.n_time == 0) || a.pf == HHFM_POOL_SUM);
  if (!all_sum || a.touch_stamp || a.pos_out || a.neg_out || a.n_neg != 10) return 1;
  if (a.K != 32 && a.K != 64 && a.K != 128) return 1;
  int dev = -1;
  cudaGetDevice(&dev);
  PgPlan* p = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_pg_mu);
    for (PgPlan* q : g_pg_plans)
      if (q->V == a.V) { p = q; break; }
  }
  if (p == nullptr || p->M != M || p->K != a.K || p->n_pool != a.n_ctx + a.n_time || p->stride != a.stride || p->device != dev)
    return 1;
  const int kv = a.K / 4;
  const int64_t rows = p->desc.row0[p->desc.n_groups];
  const int pre_grid = (int)std::min<int64_t>((rows * kv + kBlock - 1) / kBlock, (int64_t)sm_count() * 8);
  pool_groups_presum_kernel<<<pre_grid, kBlock, 0, st>>>(a.V, a.K, p->S, p->desc);
  int r = check_launch("pool_groups_presum_kernel");
  if (r != HHFM_OK) { *rc = r; return 0; }
  int miss = 1;
  switch (a.K) {
    case 32: miss = launch_pr_grouped_np<8>(a, *p, st, &r); break;
    case 64: miss = launch_pr_grouped_np<16>(a, *p, st, &r); break;
    default: miss = launch_pr_grouped_np<32>(a, *p, st, &r); break;
  }
  if (miss) return 1;                       // the planned slot count has no instance: S is rebuilt next call anyway
  if (r != HHFM_OK) { *rc = r; return 0; }
  pool_groups_expand_kernel<<<(int)p->desc.mrow0[p->desc.n_groups], kPgExpandThreads, 0, st>>>(p->G, a.K, a.gV, p->desc);
  r = check_launch("pool_groups_expand_kernel");
  if (r != HHFM_OK) { *rc = r; return 0; }
  const cudaError_t e = cudaMemsetAsync(p->G, 0, (size_t)rows * a.K * sizeof(float), st);
  if (e != cudaSuccess) {
    set_error("pool_groups: clearing G: %s", cudaGetErrorString(e));
    *rc = HHFM_ERR_LAUNCH;
    return 0;
  }
  *rc = HHFM_OK;
  return 0;
}

// ---------------------------------------------------------------------------------------------------
// Staged variant of the sum-pooling training pass for tables that do not fit in L2 (scaled config: M = 10^7, K = 128,
// 5 GB of rows; every gathered row comes from HBM).  Same per-warp pipeline as fm_train_staged_kernel (fm.cu): iteration t
//   (A) LDGSTS the W = 2 + NP + NNEG ids of sample t                                  -> id ring
//   (B) sample t-PD: one bulk copy (cp.async.bulk, UBLKCP) per row, lane w copies row w -> row stage, completion on the
//       stage's mbarrier; LDGSTS of hot_slot[id]                                         -> per-stage side buffer
//   (C) sample t-PD-NS+1: wait on its mbarrier, forward + loss + backward from shared memory, REDs from registers
// so NS*W rows (20 KB at W = 20, K = 128, NS = 2) are in flight per warp at no register cost.  One sample per warp
// iteration; lane l owns the float4 columns l, l+32, ...  Arithmetic order as in pairrank_sum_train_kernel (the idle upper
// lanes of K < 128 add exact zeros to the butterfly sums).  Touched rows are marked with a plain store into the stamp array
// and compacted afterwards (launch_touched_compact) instead of one returning atomic per row.
// ---------------------------------------------------------------------------------------------------
constexpr int kPrStagedWarps = 10;
constexpr int kPrMaxW = 32;

// shared memory per warp: NS row stages [W][K] floats, then (NS+PD) id slots and NS hot-slot slots of kPrMaxW words each,
// then NS mbarriers.
__host__ __device__ inline size_t pr_staged_warp_bytes(int NS, int W, int K) {
  const int PD = NS - 1;
  const size_t b = (size_t)NS * W * K * 4 + (size_t)((NS + PD) + NS) * kPrMaxW * 4 + (size_t)NS * 8;
  return (b + 127) / 128 * 128;
}

template <int NS, int NW = kPrStagedWarps>
__global__ void __launch_bounds__(NW * 32, 1) pairrank_sum_train_staged_kernel(const PrArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ float scratch[32];
  constexpr int PD = NS - 1;
  constexpr int RI = NS + PD;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int NP = a.n_ctx + a.n_time, NNEG = a.n_neg;
  const int W = 2 + NP + NNEG;
  const int K = a.K, kv = K >> 2;
  const uint32_t row_bytes = (uint32_t)K * 4u;
  unsigned char* base = smem_raw + (size_t)warp * pr_staged_warp_bytes(NS, W, K);
  float* rows = reinterpret_cast<float*>(base);                                   // [NS][W][K]
  int* idring = reinterpret_cast<int*>(base + (size_t)NS * W * K * 4);             // [RI][32]
  int* slotbuf = idring + RI * kPrMaxW;                                            // [NS][32]
  uint64_t* bars = reinterpret_cast<uint64_t*>(slotbuf + NS * kPrMaxW);            // [NS]
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NS; i++) mbar_init1(bars + i);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncwarp();

  const int64_t n_warps = (int64_t)gridDim.x * NW;
  const int64_t warp_g = (int64_t)blockIdx.x * NW + warp;
  const int64_t per = (a.B + n_warps - 1) / n_warps;
  const int64_t s_beg = warp_g * per;
  const int64_t s_end = (s_beg + per < a.B) ? s_beg + per : a.B;
  const int64_t n = s_end > s_beg ? s_end - s_beg : 0;
  const int rep = a.hot.slot ? (int)(warp_g % a.hot.n_rep) : 0;
  float loss_acc = 0.f;

  for (int64_t t = 0; t < n + PD + NS - 1; t++) {
    if (t < n && lane < W) ldgsts4(idring + (t % RI) * kPrMaxW + lane, a.idx + (s_beg + t) * a.stride + lane);
    ldgsts_wait<(PD > 0 ? PD - 1 : 0)>();      // groups <= t-PD complete: ids of sample t-PD, hot slots of the consumed sample
    __syncwarp();
    const int64_t j = t - PD;
    if (j >= 0 && j < n) {
      const int st = (int)(j % NS);
      if (lane == 0) mbar_expect(bars + st, row_bytes * (uint32_t)W);
      __syncwarp();
      if (lane < W) {
        const int id = idring[(j % RI) * kPrMaxW + lane];
        bulk_row(rows + ((size_t)st * W + lane) * K, a.V + (size_t)id * K, row_bytes, bars + st);
        if (a.hot.slot) ldgsts4(slotbuf + st * kPrMaxW + lane, a.hot.slot + id);
      }
    }
    ldgsts_commit();
    const int64_t c = t - PD - NS + 1;
    if (c >= 0 && c < n) {
      const int st = (int)(c % NS);
      mbar_wait_parity(bars + st, (uint32_t)((c / NS) & 1));
      const float4* r4 = reinterpret_cast<const float4*>(rows + (size_t)st * W * K);
      const int* ids = idring + (c % RI) * kPrMaxW;
      const int* slots = slotbuf + st * kPrMaxW;
      float4 hyb[4];
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const int cc = lane + 32 * i;
        hyb[i] = f4_zero();
        if (cc < kv) {
          hyb[i] = r4[cc];                                       // user, then ctx.., time.. in record order
          for (int q = 0; q < NP; q++) hyb[i] = f4_add(hyb[i], r4[(2 + q) * kv + cc]);
        }
      }
      auto dot_row = [&](int w) {
        float p = 0.f;
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int cc = lane + 32 * i;
          if (cc < kv) p += f4_dot(hyb[i], r4[w * kv + cc]);
        }
        return warp_sum(p);
      };
      const float pos = dot_row(1);
      float m = -INFINITY;
      unsigned tie = 0u;
      for (int jn = 0; jn < NNEG; jn++) {
        const float p = dot_row(2 + NP + jn);
        if (p > m) { m = p; tie = 1u << jn; }
        else if (p == m) tie |= 1u << jn;
      }
      const float x = pos - m;
      const float sg = 1.f / (1.f + expf(-x));
      if (lane == 0) loss_acc += -logf(sg);
      const float gp = sg - 1.f;
      const float gn = -gp / (float)__popc(tie);
      auto dst_of = [&](int w) {
        const int slot = a.hot.slot ? slots[w] : -1;
        return (slot >= 0) ? a.hot.ghot + ((size_t)rep * a.hot.n_hot + slot) * K : a.gV + (size_t)ids[w] * K;
      };
      float4 dh[4];
      {
        float* d = dst_of(1);
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int cc = lane + 32 * i;
          if (cc < kv) {
            dh[i] = f4_scale(r4[kv + cc], gp);
            red_add_v4(d + 4 * cc, f4_scale(hyb[i], gp));
          }
        }
      }
      unsigned wl = tie;
      while (wl) {
        const int jn = __ffs((int)wl) - 1;
        wl &= wl - 1;
        const int w = 2 + NP + jn;
        float* d = dst_of(w);
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int cc = lane + 32 * i;
          if (cc < kv) {
            dh[i] = f4_fma(r4[w * kv + cc], gn, dh[i]);
            red_add_v4(d + 4 * cc, f4_scale(hyb[i], gn));
          }
        }
      }
      for (int w = 0; w < 2 + NP; w++) {
        if (w == 1) continue;
        float* d = dst_of(w);
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int cc = lane + 32 * i;
          if (cc < kv) red_add_v4(d + 4 * cc, dh[i]);
        }
      }
      if (a.touch_stamp && lane < W) {
        const bool touched = (lane < 2 + NP) || ((tie >> (lane - 2 - NP)) & 1u);
        if (touched) a.touch_stamp[ids[lane]] = a.stamp;       // compacted into the list afterwards
      }
      __syncwarp();     // every lane is done with this stage before the next iteration re-arms it
    }
  }
  ldgsts_wait<0>();
  const float bl = block_sum(loss_acc, scratch);
  write_partial(a.loss_partials, bl);
}

// HHFM_ERR_UNSUPPORTED when the configuration is not covered or the table is small enough to live in L2 (the register
// kernel wins there).  HHFM_PR_STAGED=0/1 forces the choice.
static int dispatch_pr_staged(const PrArgs& a, int64_t M, cudaStream_t st) {
  const bool all_sum = (a.n_ctx == 0 || a.pc == HHFM_POOL_SUM) && (a.n_time == 0 || a.pt == HHFM_POOL_SUM) &&
                       ((a.n_ctx == 0 && a.n_time == 0) || a.pf == HHFM_POOL_SUM);
  if (!all_sum || a.pos_out || a.neg_out) return HHFM_ERR_UNSUPPORTED;
  const int W = 2 + a.n_ctx + a.n_time + a.n_neg;
  if (W > kPrMaxW || a.n_neg < 1 || a.n_neg > 31 || a.K < 64 || a.K > 512 || W > a.stride) return HHFM_ERR_UNSUPPORTED;
  const char* env = getenv("HHFM_PR_STAGED");
  const int force = env ? (env[0] == '1' ? 1 : 0) : 2;
  if (force == 0) return HHFM_ERR_UNSUPPORTED;
  if (force == 2 && (size_t)M * a.K * 4 < ((size_t)96 << 20)) return HHFM_ERR_UNSUPPORTED;
  const size_t cap = (size_t)224 * 1024;
  int ns = 4, nw = kPrStagedWarps;
  const char* enw = getenv("HHFM_PR_WARPS");               // 7 .. 10 warps per CTA (A/B runs)
  if (enw) { const int v = atoi(enw); if (v >= 7 && v <= 10) nw = v; }
  const char* ens = getenv("HHFM_PR_STAGES");
  if (ens && ens[0] >= '2' && ens[0] <= '4') ns = ens[0] - '0';
  while (ns > 2 && pr_staged_warp_bytes(ns, W, a.K) * nw > cap) ns--;
  const size_t smem = pr_staged_warp_bytes(ns, W, a.K) * nw;
  if (smem > cap) return HHFM_ERR_UNSUPPORTED;
  const int grid = sm_count();
  if (grid > kPartials) return HHFM_ERR_UNSUPPORTED;
  cudaError_t e = cudaSuccess;
#define HHFM_LAUNCH_PR(NS_, NW_)                                                                                                  \
  do {                                                                                                                            \
    e = cudaFuncSetAttribute(pairrank_sum_train_staged_kernel<NS_, NW_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    if (e == cudaSuccess) pairrank_sum_train_staged_kernel<NS_, NW_><<<grid, NW_ * 32, smem, st>>>(a);                             \
  } while (0)
#define HHFM_LAUNCH_PR_NS(NW_)                                                                                                    \
  do {                                                                                                                            \
    if (ns == 4) HHFM_LAUNCH_PR(4, NW_);                                                                                          \
    else if (ns == 3) HHFM_LAUNCH_PR(3, NW_);                                                                                     \
    else HHFM_LAUNCH_PR(2, NW_);                                                                                                  \
  } while (0)
  if (nw == 7) HHFM_LAUNCH_PR_NS(7);
  else if (nw == 8) HHFM_LAUNCH_PR_NS(8);
  else if (nw == 9) HHFM_LAUNCH_PR_NS(9);
  else HHFM_LAUNCH_PR_NS(10);
#undef HHFM_LAUNCH_PR_NS
#undef HHFM_LAUNCH_PR
  if (e != cudaSuccess) {
    set_error("pairrank_sum_train_staged_kernel: %s", cudaGetErrorString(e));
    return HHFM_ERR_LAUNCH;
  }
  int rc = check_launch("pairrank_sum_train_staged_kernel");
  if (rc != HHFM_OK) return rc;
  if (a.touch_stamp != nullptr) rc = launch_touched_compact(a.touch_stamp, a.stamp, M, a.touched_rows, a.touched_count, st);
  return rc;
}

template <int LPS, int VPL, int MODE, bool ANYMAX>
static int launch_pr(const PrArgs& a, int deterministic, cudaStream_t st) {
  static int occ = 0;
  if (occ == 0) {
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pairrank_kernel<LPS, VPL, MODE, ANYMAX>, kBlock, 0);
    if (occ < 1) occ = 1;
  }
  PrArgs b = a;
  constexpr int G = 32 / LPS;
  if (deterministic) {
    b.groups_active = 1;
    pairrank_kernel<LPS, VPL, MODE, ANYMAX><<<1, 32, 0, st>>>(b);
  } else {
    b.groups_active = G;
    const int grid = grid_for(a.B, (kBlock / 32) * G, occ);
    pairrank_kernel<LPS, VPL, MODE, ANYMAX><<<grid, kBlock, 0, st>>>(b);
  }
  return check_launch("pairrank_kernel");
}

template <int MODE>
static int dispatch_pr(const PrArgs& a, int deterministic, cudaStream_t st) {
  const bool anymax = (a.n_ctx > 0 && a.pc == HHFM_POOL_MAX) || (a.n_time > 0 && a.pt == HHFM_POOL_MAX) ||
                      ((a.n_ctx > 0 || a.n_time > 0) && a.pf == HHFM_POOL_MAX);
  if (anymax) {
#define CALL(L, V) return launch_pr<L, V, MODE, true>(a, deterministic, st)
    HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  } else {
#define CALL(L, V) return launch_pr<L, V, MODE, false>(a, deterministic, st)
    HHFM_DISPATCH_K(a.K, CALL);
#undef CALL
  }
  return HHFM_ERR_UNSUPPORTED;
}

// HHFM_NO_FAST=1 forces the generic kernel (A/B measurements, tests of both paths).
static bool hhfm_fast_path_enabled() {
  const char* e = getenv("HHFM_NO_FAST");
  return !(e && e[0] == '1');
}

static int check_pr(const int32_t* idx, int64_t B, int64_t stride, int n_ctx, int n_time, int n_neg, int pc, int pt,
                    int pf, const float* V, int64_t M, int64_t K) {
  HHFM_REQUIRE(idx && V, "pairrank: idx and V must not be NULL");
  HHFM_REQUIRE(B >= 0 && M > 0, "pairrank: bad sizes");
  HHFM_REQUIRE(K > 0 && K % 4 == 0 && K <= 512, "pairrank: K=%lld unsupported (need K %% 4 == 0, K <= 512)", (long long)K);
  HHFM_REQUIRE(n_ctx >= 0 && n_time >= 0 && n_neg >= 0 && n_neg <= 64, "pairrank: need 0 <= n_neg <= 64, n_ctx,n_time >= 0");
  HHFM_REQUIRE(stride >= 2 + n_ctx + n_time + n_neg && stride % 4 == 0, "pairrank: stride %lld too small or not a multiple of 4", (long long)stride);
  HHFM_REQUIRE(pc >= 0 && pc <= 2 && pt >= 0 && pt <= 2 && pf >= 0 && pf <= 2, "pairrank: bad pool mode");
  HHFM_REQUIRE(((uintptr_t)V & 15) == 0 && ((uintptr_t)idx & 15) == 0, "pairrank: V and idx must be 16-byte aligned");
  return HHFM_OK;
}

static PrArgs make_args(const int32_t* idx, int64_t B, int64_t stride, int n_ctx, int n_time, int n_neg, int pc, int pt,
                        int pf, const float* V, int64_t K) {
  PrArgs a{};
  a.idx = idx; a.B = B; a.stride = (int)stride; a.n_ctx = n_ctx; a.n_time = n_time; a.n_neg = n_neg;
  a.pc = pc; a.pt = pt; a.pf = pf; a.V = V; a.K = (int)K;
  return a;
}

}  // namespace hhfm

using namespace hhfm;

extern "C" int hhfm_pairrank_fwd(const int32_t* idx, int64_t B, int64_t stride, int32_t n_ctx, int32_t n_time,
                                 int32_t n_neg, int32_t pool_ctx, int32_t pool_time, int32_t pool_stack, const float* V,
                                 int64_t M, int64_t K, float* pos_out, float* neg_out, hhfm_stream_t stream) {
  int rc = check_pr(idx, B, stride, n_ctx, n_time, n_neg, pool_ctx, pool_time, pool_stack, V, M, K);
  if (rc) return rc;
  HHFM_REQUIRE(pos_out != nullptr, "pairrank_fwd: pos_out is NULL");
  if (B == 0) return HHFM_OK;
  PrArgs a = make_args(idx, B, stride, n_ctx, n_time, n_neg, pool_ctx, pool_time, pool_stack, V, K);
  a.pos_out = pos_out; a.neg_out = neg_out;
  return dispatch_pr<PR_FWD>(a, 0, (cudaStream_t)stream);
}

extern "C" int hhfm_pairrank_fwd_bwd(const int32_t* idx, int64_t B, int64_t stride, int32_t n_ctx, int32_t n_time,
                                     int32_t n_neg, int32_t pool_ctx, int32_t pool_time, int32_t pool_stack,
                                     const float* V, int64_t M, int64_t K, float* pos_out, float* neg_out, float* gV,
                                     float* loss_partials, int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows,
                                     int32_t* touched_count, const int32_t* hot_slot, float* ghot, int32_t n_rep,
                                     int32_t n_hot, int32_t deterministic, hhfm_stream_t stream) {
  int rc = check_pr(idx, B, stride, n_ctx, n_time, n_neg, pool_ctx, pool_time, pool_stack, V, M, K);
  if (rc) return rc;
  HHFM_REQUIRE(!hot_slot || (ghot && n_rep >= 1 && n_hot >= 1), "pairrank_fwd_bwd: hot_slot needs ghot, n_rep, n_hot");
  HHFM_REQUIRE(B > 0 && n_neg >= 1, "pairrank_fwd_bwd: needs B > 0 and at least one negative");
  HHFM_REQUIRE(gV && loss_partials, "pairrank_fwd_bwd: gV and loss_partials are required");
  HHFM_REQUIRE(!touch_stamp || (touched_rows && touched_count), "pairrank_fwd_bwd: touch_stamp needs touched_rows/count");
  HHFM_REQUIRE(((uintptr_t)gV & 15) == 0, "pairrank: gV must be 16-byte aligned");
  PrArgs a = make_args(idx, B, stride, n_ctx, n_time, n_neg, pool_ctx, pool_time, pool_stack, V, K);
  a.pos_out = pos_out; a.neg_out = neg_out; a.gV = gV; a.loss_partials = loss_partials;
  a.touch_stamp = touch_stamp; a.stamp = stamp; a.touched_rows = touched_rows; a.touched_count = touched_count;
  a.hot = HotPlan{hot_slot, ghot, nullptr, n_rep, n_hot};
  if (!deterministic && hhfm_fast_path_enabled()) {
    int frc = dispatch_pr_staged(a, M, (cudaStream_t)stream);
    if (frc != HHFM_ERR_UNSUPPORTED) return frc;
    if (dispatch_pr_grouped(a, M, (cudaStream_t)stream, &frc) == 0) return frc;
    if (dispatch_pr_fast(a, (cudaStream_t)stream, &frc) == 0) return frc;
  }
  return dispatch_pr<PR_TRAIN>(a, deterministic, (cudaStream_t)stream);
}

extern "C" int hhfm_pool_groups_attach(const float* V, int64_t M, int64_t K, int32_t n_pool, int64_t stride,
                                       const int32_t* col_group, const int32_t* col_lo, const int32_t* col_card,
                                       int64_t* handle) {
  HHFM_REQUIRE(V && col_group && col_lo && col_card && handle, "pool_groups_attach: NULL argument");
  HHFM_REQUIRE(K == 32 || K == 64 || K == 128, "pool_groups_attach: K=%lld unsupported (32, 64, 128)", (long long)K);
  HHFM_REQUIRE(n_pool == 3 || n_pool == 8 || n_pool == 10, "pool_groups_attach: n_pool=%d unsupported (3, 8, 10)", n_pool);
  HHFM_REQUIRE(M > 0 && stride >= 2 + n_pool && stride % 4 == 0, "pool_groups_attach: bad sizes");
  PgPlan* p = new PgPlan{};
  p->V = V; p->M = M; p->K = (int)K; p->n_pool = n_pool; p->stride = (int)stride;
  cudaGetDevice(&p->device);
  int group_slot[kPgMaxCols];
  int n_groups = 0, n_slots = 0;
  for (int c = 0; c < kPgMaxCols; c++) group_slot[c] = -1;
  PgDesc& d = p->desc;
  int grp_of_slot[kPgMaxSlots];
  bool ok = true;
  for (int c = 0; c < n_pool && ok; c++) {
    const int gid = col_group[c];
    if (gid < 0) {
      if (n_slots == kPgMaxSlots) { ok = false; break; }
      p->pg.slot_of[c] = n_slots; p->pg.lo[c] = 0; p->pg.card[c] = 0xffffffffu; p->pg.mult[c] = 1;
      p->pg.T[n_slots] = V; p->pg.G[n_slots] = nullptr;
      n_slots++;
      continue;
    }
    if (gid >= n_pool || col_card[c] < 1 || col_lo[c] < 0 || (int64_t)col_lo[c] + col_card[c] > M) { ok = false; break; }
    if (group_slot[gid] < 0) {
      if (n_slots == kPgMaxSlots) { ok = false; break; }
      group_slot[gid] = n_slots;
      grp_of_slot[n_slots] = n_groups;
      d.n_mem[n_groups] = 0;
      n_groups++;
      n_slots++;
    }
    const int s = group_slot[gid], g = grp_of_slot[s];
    p->pg.slot_of[c] = s; p->pg.lo[c] = col_lo[c]; p->pg.card[c] = (unsigned)col_card[c];
    d.mem_lo[g][d.n_mem[g]] = col_lo[c];
    d.mem_card[g][d.n_mem[g]] = col_card[c];
    d.n_mem[g]++;
  }
  // mixed-radix weights (members in record order), table rows, member rows
  d.n_groups = n_groups;
  d.row0[0] = 0; d.mrow0[0] = 0;
  for (int g = 0; g < n_groups && ok; g++) {
    int64_t P = 1, mr = 0;
    for (int m = 0; m < d.n_mem[g]; m++) { P *= d.mem_card[g][m]; mr += d.mem_card[g][m]; if (P > (1 << 24)) ok = false; }
    d.row0[g + 1] = d.row0[g] + P;
    d.mrow0[g + 1] = d.mrow0[g] + mr;
  }
  for (int c = 0; c < n_pool && ok; c++) {
    if (col_group[c] < 0) continue;
    const int s = p->pg.slot_of[c];
    int mult = 1;
    for (int c2 = 0; c2 < c; c2++)
      if (col_group[c2] >= 0 && p->pg.slot_of[c2] == s) mult *= col_card[c2];
    p->pg.mult[c] = mult;
    for (int c2 = c + 1; c2 < n_pool; c2++)          // member rows of different columns must not overlap
      if (col_group[c2] >= 0 && col_lo[c2] < col_lo[c] + col_card[c] && col_lo[c] < col_lo[c2] + col_card[c2]) ok = false;
  }
  const int max_slots = n_pool == 3 ? 2 : kPgMaxSlots;   // compiled instances: NS < NP, NS <= 4
  if (!ok || n_groups == 0 || n_slots > max_slots || d.row0[n_groups] > (1 << 24)) {
    delete p;
    set_error("pool_groups_attach: the plan is not supported (at most %d pooled rows, at least one group, group ranges "
              "inside [0, M) and disjoint, at most 2^24 combinations)", max_slots);
    return HHFM_ERR_BAD_ARG;
  }
  p->n_slots = n_slots;
  const size_t bytes = (size_t)d.row0[n_groups] * K * sizeof(float);
  cudaError_t e = cudaMalloc(&p->S, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&p->G, bytes);
  if (e == cudaSuccess) e = cudaMemset(p->G, 0, bytes);
  if (e != cudaSuccess) {
    pg_free(p);
    set_error("pool_groups_attach: %s", cudaGetErrorString(e));
    return HHFM_ERR_LAUNCH;
  }
  for (int s = 0; s < n_slots; s++)
    if (p->pg.T[s] == nullptr) {                   // group slot
      p->pg.T[s] = p->S + (size_t)d.row0[grp_of_slot[s]] * K;
      p->pg.G[s] = p->G + (size_t)d.row0[grp_of_slot[s]] * K;
    }
  std::lock_guard<std::mutex> lk(g_pg_mu);
  for (size_t i = 0; i < g_pg_plans.size(); i++)
    if (g_pg_plans[i]->V == V) {                   // a new plan for the same table replaces the old one
      pg_free(g_pg_plans[i]);
      g_pg_plans.erase(g_pg_plans.begin() + i);
      break;
    }
  p->handle = g_pg_next++;
  g_pg_plans.push_back(p);
  *handle = p->handle;
  return HHFM_OK;
}

extern "C" int hhfm_pool_groups_detach(const float* V, int64_t handle) {
  std::lock_guard<std::mutex> lk(g_pg_mu);
  for (size_t i = 0; i < g_pg_plans.size(); i++)
    if (g_pg_plans[i]->V == V && g_pg_plans[i]->handle == handle) {
      pg_free(g_pg_plans[i]);
      g_pg_plans.erase(g_pg_plans.begin() + i);
      break;
    }
  return HHFM_OK;
}

extern "C" int hhfm_pool_groups_tables(const float* V, float** S, float** G, int64_t* rows) {
  HHFM_REQUIRE(S && G && rows, "pool_groups_tables: NULL argument");
  std::lock_guard<std::mutex> lk(g_pg_mu);
  for (PgPlan* p : g_pg_plans)
    if (p->V == V) {
      *S = p->S; *G = p->G; *rows = p->desc.row0[p->desc.n_groups];
      return HHFM_OK;
    }
  set_error("pool_groups_tables: no plan is attached to this table");
  return HHFM_ERR_BAD_ARG;
}

extern "C" int hhfm_pairrank_bwd(const int32_t* idx, int64_t B, int64_t stride, int32_t n_ctx, int32_t n_time,
                                 int32_t n_neg, int32_t pool_ctx, int32_t pool_time, int32_t pool_stack, const float* V,
                                 int64_t M, int64_t K, const float* dpos, const float* dneg, float* gV,
                                 int32_t deterministic, hhfm_stream_t stream) {
  int rc = check_pr(idx, B, stride, n_ctx, n_time, n_neg, pool_ctx, pool_time, pool_stack, V, M, K);
  if (rc) return rc;
  HHFM_REQUIRE(dpos && gV, "pairrank_bwd: dpos and gV are required");
  if (B == 0) return HHFM_OK;
  PrArgs a = make_args(idx, B, stride, n_ctx, n_time, n_neg, pool_ctx, pool_time, pool_stack, V, K);
  a.dpos = dpos; a.dneg = dneg; a.gV = gV;
  return dispatch_pr<PR_BWD>(a, deterministic, (cudaStream_t)stream);
}
