// Data-parallel training step (SURVEY.md 8e): hot-replica fold + cross-GPU gradient all-reduce + TF1 optimizer + loss
// reduction as ONE persistent kernel, `dp_step_kernel`.
//
// Every rank owns an exchange buffer X in symmetric memory (same size on every rank, mapped into every peer, and -- on an
// NVSwitch box -- bound to one multicast object; the allocation and the address exchange are torch.distributed plumbing,
// hhfm_b200/dist.py).  The flat gradient index space is cut into pieces of 32 float4 (512 bytes); piece p belongs to rank
// p % N for the reduction and to CTA (p / N) % G on EVERY rank for everything else, so all dependencies are between the
// CTAs with the same index on the N ranks -- there is no grid-wide barrier anywhere in the kernel.  CTA b of rank r:
//
//   A  its pieces: arena (+ the hot-row replicas of those elements, fixed replica order) -> X, arena and replicas cleared
//   -- flag exchange with CTA b of every other rank (system-scope release / acquire flags in symmetric memory)
//   B  its pieces that rank r owns: sum over all ranks -- `multimem.ld_reduce` (the NVSwitch adds the ranks' copies in
//      flight) or, without a multicast mapping, peer loads in rank order -- written back into EVERY rank's X
//      (`multimem.st` / peer stores).  All replicas therefore consume the same bits and stay bit-identical.
//   -- flag exchange with CTA b of every other rank
//   C  its pieces: g = X (local), g_eff = g + lamda*w, optimizer update of the local replica (same expressions as opt.cu),
//      sum of w^2 for the regulariser; the last CTA to finish adds up the loss.
//
// With n_ranks == 1 the exchange drops out (A feeds C through registers) and the kernel is the single-GPU tail of a step
// (fold + optimizer + loss in one launch instead of three).  The flag waits are bounded: on a timeout the kernel raises a
// sticky error flag in device memory (read back by the host together with the loss) and every later step returns
// immediately -- the CUDA context stays usable (no __trap).  The launch is cooperative only for its guarantee that all
// CTAs are resident (a CTA waits for its peers on other GPUs, never for a CTA of its own grid).
#include <cooperative_groups.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace hhfm {

constexpr int kMaxPeers = 16;
constexpr int kMaxSegs = 4;
constexpr int kDpThreads = 512;

struct DpSeg {
  float* w;
  float* s1;
  float* s2;
  int64_t off;   // gradient of w[0, n) = X[off, off + n)
  int64_t n;
  float lamda;
  int width;     // hhfm_dp_step_touched: row width of an IndexedSlices variable (only touched rows move), 0 = dense
};

struct OptP2 {
  float lr, lamda, b1, b2, eps;   // adagrad: lr; adam: lr_t, b1, b2, eps; momentum: lr, b1 = momentum; sgd: lr
};

struct DpArgs {
  DpSeg seg[kMaxSegs];
  int n_seg;
  float* arena;          // rank-private gradient arena, n_g floats used (16-byte aligned, readable up to roundup4(n_g))
  int64_t n_g;
  float* ghot;           // hot-row replicas [n_rep, n_hot, K] (+ bias [n_rep, n_hot]) or NULL
  float* ghot_bias;
  int n_rep, n_hot, K;
  const int32_t* hot_slot;   // [M] slot of a table row or -1
  int64_t M;                 // table rows: the table gradient is arena[0, M*K)
  int64_t bias_off;          // offset of the feature_bias gradient inside the arena (used with ghot_bias)
  const float* loss_partials;
  float* x;              // this rank's exchange buffer: roundup4(n_g) gradient floats + one float4 whose .x is the loss
  float* x_mc;           // multicast alias of X or NULL
  float* x_peer[kMaxPeers];
  int32_t* flag_peer[kMaxPeers];   // flag arrays (2 * gridDim.x * kMaxPeers int32 each) of every rank, own one included
  int rank, n_ranks;
  int32_t* state;        // device: [0] step counter, [1] sticky error, [2] finished-CTA ticket
  OptP2 p;
  float* sq_ws;          // [gridDim.x + 1] per-CTA regulariser partials, then the all-rank data loss
  float* loss_out;
  long long timeout_cycles;
  int fences;            // 1: explicit system fences around the flag release / acquire (HHFM_DP_FENCES, A/B)
  const int32_t* stamps; // hhfm_dp_step_touched: [M] touched-row stamps of this rank's scatter kernels
  int32_t stamp;         //   the current step's stamp
};

// same expressions as opt.cu::opt_elem, so the fused step is bit-identical to the separate optimizer kernel
template <int KIND>
__device__ __forceinline__ void opt_elem2(float& w, float& a, float& b, float g, const OptP2& p) {
  if (KIND == HHFM_OPT_ADAGRAD) {
    a = fmaf(g, g, a);
    w = w - p.lr * g / sqrtf(a);
  } else if (KIND == HHFM_OPT_ADAM) {
    a = fmaf(p.b1, a, (1.f - p.b1) * g);              // explicit contraction: the same bits in every kernel that inlines this
    b = fmaf(p.b2, b, (1.f - p.b2) * (g * g));
    w = w - p.lr * a / (sqrtf(b) + p.eps);
  } else if (KIND == HHFM_OPT_MOMENTUM) {
    a = fmaf(a, p.b1, g);
    w = fmaf(-p.lr, a, w);
  } else {
    w = fmaf(-p.lr, g, w);
  }
}

__device__ __forceinline__ float4 ld_cv4(const float4* p) { return __ldcv(p); }   // never a stale L1 line

__device__ __forceinline__ float4 multimem_ld_reduce4(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(mc)
               : "memory");
  return v;
}

__device__ __forceinline__ void multimem_st4(float* mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// Executed by warp 0 of a CTA after a __syncthreads(): lane r publishes `value` into rank r's flag slot of this CTA and
// waits for rank r's value in the local array.  Returns false on a timeout.
__device__ __forceinline__ bool cross_rank_flags(const DpArgs& a, int phase, int32_t value) {
  const int r = threadIdx.x;
  bool ok = true;
  if (r < a.n_ranks) {
    const int slot = (phase * (int)gridDim.x + (int)blockIdx.x) * kMaxPeers;
    if (a.fences) __threadfence_system();
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(a.flag_peer[r] + slot + a.rank), "r"(value) : "memory");
    const int32_t* mine = a.flag_peer[a.rank] + slot + r;
    const long long t0 = clock64();
    for (;;) {
      int32_t v;
      asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
      if (v - value >= 0) break;
      if (clock64() - t0 > a.timeout_cycles) {
        ok = false;
        break;
      }
    }
    if (a.fences) __threadfence_system();
  }
  return ok;
}

constexpr int kPiece = 32;      // float4 per piece (512 bytes)

// TOUCHED (hhfm_dp_step_touched): segments with a row width move only the rows stamped on SOME rank.  Every float of a
// piece has one bit in a 4-word mask stored behind the gradient floats of X (piece p: words 4p .. 4p+3, lane l's float4 in
// bits 4(l%8) .. 4(l%8)+3 of word l/8).  A: each rank writes the bits of its local stamps; B: the owner ORs the ranks'
// masks together with the piece sum; C: the update reads the OR.  The bit of a float is the stamp of its row, so a row that
// straddles two pieces gets the same decision in both.
template <int KIND, bool TOUCHED>
__global__ void __launch_bounds__(kDpThreads) dp_step_kernel(const DpArgs a) {
  __shared__ float scratch[32];
  __shared__ float s_loss;
  __shared__ int s_last;
  const int G = (int)gridDim.x, b = (int)blockIdx.x, N = a.n_ranks;
  const int lane = threadIdx.x & 31, pslot = threadIdx.x >> 5;
  constexpr int kSlots = kDpThreads / 32;            // pieces a CTA works on per iteration
  const int32_t step = __ldcv(a.state);
  if (__ldcv(a.state + 1) != 0) return;              // sticky error of an earlier step

  const int64_t n_g4 = (a.n_g + 3) >> 2;             // gradient float4; element n_g4 is the loss slot
  const int64_t total4 = n_g4 + 1;
  const int64_t n_pieces = (total4 + kPiece - 1) / kPiece;
  const int64_t nv4 = (a.M * (int64_t)a.K) >> 2;
  const int kv = a.K >> 2;
  const int64_t p_loss = n_g4 / kPiece;
  const bool owns_loss = ((p_loss / N) % G) == b;
  float4* arena4 = reinterpret_cast<float4*>(a.arena);
  float4* x4 = reinterpret_cast<float4*>(a.x);
  uint32_t* xmask = reinterpret_cast<uint32_t*>(x4 + total4);      // TOUCHED, n_ranks > 1: [n_pieces][4] words

  // this rank's data loss (sum of the per-CTA partials of the scatter kernel), by the CTA that owns the loss slot
  if (owns_loss) {                                   // CTA-uniform; all threads: four independent loads each, not 64 in a chain
    float l = 0.f;
#pragma unroll
    for (int i = 0; i < kPartials / kDpThreads; i++) l += __ldcv(a.loss_partials + threadIdx.x + i * kDpThreads);
    l = block_sum(l, scratch);
    if (threadIdx.x == 0) s_loss = l;
  }
  __syncthreads();

  // element i of my pieces, in a fixed order: local piece L -> piece ((L / N) * G + b) * N + L % N
  auto piece_of = [&](int64_t L) { return ((L / N) * G + b) * N + (L % N); };

  // arena element i with its hot-row replicas folded in (replica order fixed: reproducible); arena and replicas are cleared
  auto take = [&](int64_t i) {
    if (i == n_g4) return make_float4(s_loss, 0.f, 0.f, 0.f);
    float4 v = arena4[i];
    arena4[i] = f4_zero();
    if (a.ghot != nullptr) {
      if (i < nv4) {
        const int s = __ldg(a.hot_slot + i / kv);
        if (s >= 0) {
          const int c = (int)(i % kv);
          constexpr int kFoldBatch = 16;            // replica loads in flight per thread (the fold is the long pole of phase A)
          for (int r0 = 0; r0 < a.n_rep; r0 += kFoldBatch) {
            float4 t[kFoldBatch];
#pragma unroll
            for (int q = 0; q < kFoldBatch; q++) {
              float4* p = reinterpret_cast<float4*>(a.ghot + ((size_t)(r0 + q) * a.n_hot + s) * a.K) + c;
              t[q] = (r0 + q < a.n_rep) ? *p : f4_zero();
            }
#pragma unroll
            for (int q = 0; q < kFoldBatch; q++) {
              if (r0 + q < a.n_rep) {
                v = f4_add(v, t[q]);
                *(reinterpret_cast<float4*>(a.ghot + ((size_t)(r0 + q) * a.n_hot + s) * a.K) + c) = f4_zero();
              }
            }
          }
        }
      } else if (a.ghot_bias != nullptr) {
        float* vv = reinterpret_cast<float*>(&v);
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const int64_t f = 4 * i + j - a.bias_off;
          if (f < 0 || f >= a.M) continue;
          const int s = __ldg(a.hot_slot + f);
          if (s < 0) continue;
          float acc = 0.f;
          for (int r0 = 0; r0 < a.n_rep; r0 += 16) {        // 16 loads in flight, added in replica order
            float t[16];
#pragma unroll
            for (int q = 0; q < 16; q++) t[q] = (r0 + q < a.n_rep) ? a.ghot_bias[(size_t)(r0 + q) * a.n_hot + s] : 0.f;
#pragma unroll
            for (int q = 0; q < 16; q++) {
              if (r0 + q < a.n_rep) {
                acc += t[q];
                a.ghot_bias[(size_t)(r0 + q) * a.n_hot + s] = 0.f;
              }
            }
          }
          vv[j] += acc;
        }
      }
    }
    return v;
  };

  // optimizer update of the (up to four) parameters whose gradient is flat element i; returns the regulariser share
  // the touched bits (bit j: float 4i+j) of flat element i from this rank's stamps
  auto local_bits = [&](int64_t i) {
    uint32_t m = 0;
    if (!TOUCHED || i >= n_g4) return m;
    for (int sgi = 0; sgi < a.n_seg; sgi++) {
      const DpSeg& sg = a.seg[sgi];
      if (sg.width == 0) continue;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int64_t e = 4 * i + j - sg.off;
        if (e >= 0 && e < sg.n && __ldg(a.stamps + e / sg.width) == a.stamp) m |= 1u << j;
      }
    }
    return m;
  };

  // optimizer update of the (up to four) parameters whose gradient is flat element i; returns the regulariser share.
  // TOUCHED: a float of a segment with a row width moves only if its bit in `tbits` is set, with g_eff = g (no L2 term),
  // as in opt.cu::opt_rows_kernel
  auto apply = [&](int64_t i, float4 gv, uint32_t tbits) {
    float reg = 0.f;
    const int64_t f0 = 4 * i;
    for (int sgi = 0; sgi < a.n_seg; sgi++) {
      const DpSeg& sg = a.seg[sgi];
      if (f0 + 4 <= sg.off || f0 >= sg.off + sg.n) continue;
      const bool rows = TOUCHED && sg.width > 0;
      if (rows && tbits == 0) continue;
      OptP2 p = a.p;
      p.lamda = sg.lamda;
      const int64_t e0 = f0 - sg.off;
      if (e0 >= 0 && e0 + 4 <= sg.n && (e0 & 3) == 0 && (!rows || tbits == 0xFu)) {
        float4* w4 = reinterpret_cast<float4*>(sg.w + e0);
        float4* a4 = reinterpret_cast<float4*>(sg.s1 + e0);
        float4* b4 = reinterpret_cast<float4*>(sg.s2 + e0);
        float4 wv = *w4;
        float4 av = (KIND != HHFM_OPT_SGD) ? *a4 : f4_zero();
        float4 bv = (KIND == HHFM_OPT_ADAM) ? *b4 : f4_zero();
        const float sq = f4_dot(wv, wv);
        float4 ge = rows ? gv : f4_fma(wv, p.lamda, gv);
        opt_elem2<KIND>(wv.x, av.x, bv.x, ge.x, p);
        opt_elem2<KIND>(wv.y, av.y, bv.y, ge.y, p);
        opt_elem2<KIND>(wv.z, av.z, bv.z, ge.z, p);
        opt_elem2<KIND>(wv.w, av.w, bv.w, ge.w, p);
        *w4 = wv;
        if (KIND != HHFM_OPT_SGD) *a4 = av;
        if (KIND == HHFM_OPT_ADAM) *b4 = bv;
        if (sg.lamda > 0.f) reg += 0.5f * sg.lamda * sq;
        return reg;
      }
      const float* gs = reinterpret_cast<const float*>(&gv);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int64_t e = e0 + j;
        if (e < 0 || e >= sg.n) continue;
        if (rows && !((tbits >> j) & 1u)) continue;
        float wv = sg.w[e];
        float av = (KIND != HHFM_OPT_SGD) ? sg.s1[e] : 0.f;
        float bv = (KIND == HHFM_OPT_ADAM) ? sg.s2[e] : 0.f;
        if (sg.lamda > 0.f) reg += 0.5f * sg.lamda * wv * wv;
        float ge = rows ? gs[j] : fmaf(wv, p.lamda, gs[j]);
        opt_elem2<KIND>(wv, av, bv, ge, p);
        sg.w[e] = wv;
        if (KIND != HHFM_OPT_SGD) sg.s1[e] = av;
        if (KIND == HHFM_OPT_ADAM) sg.s2[e] = bv;
      }
    }
    return reg;
  };

  float reg = 0.f, loss_all = 0.f;
  bool has_loss = false;
  if (N == 1) {
    // ---- single GPU: A feeds C through registers ----
    for (int64_t L = pslot;; L += kSlots) {
      const int64_t p = piece_of(L);
      if (p >= n_pieces) break;
      const int64_t i = p * kPiece + lane;
      if (i >= total4) continue;
      const float4 v = take(i);
      if (i == n_g4) { loss_all = v.x; has_loss = true; }
      else reg += apply(i, v, local_bits(i));
    }
  } else {
    // ---- A: my pieces -> X ----
    for (int64_t L = pslot;; L += kSlots) {
      const int64_t p = piece_of(L);
      if (p >= n_pieces) break;
      const int64_t i = p * kPiece + lane;
      if (i < total4) x4[i] = take(i);
      if (TOUCHED) {
        const uint32_t nib = (i < total4) ? local_bits(i) << (4 * (lane & 7)) : 0u;
#pragma unroll
        for (int w = 0; w < 4; w++) {
          const uint32_t word = __reduce_or_sync(0xffffffffu, (lane >> 3) == w ? nib : 0u);
          if (lane == w) xmask[4 * p + w] = word;
        }
      }
    }
    // the CTA barrier orders every thread's stores before the signalling lanes, whose system-scope fence + release store is
    // cumulative over them: no per-thread system fence
    __syncthreads();
    if (threadIdx.x < 32 && !cross_rank_flags(a, 0, step + 1)) a.state[1] = 1;
    __syncthreads();
    // ---- B: all-reduce of my pieces that this rank owns (L % N == rank), result into every rank's X ----
    for (int64_t L = (int64_t)pslot * N + a.rank;; L += (int64_t)kSlots * N) {
      const int64_t p = piece_of(L);
      if (p >= n_pieces) break;
      const int64_t i = p * kPiece + lane;
      if (TOUCHED && lane < 4) {                     // the piece's touched mask: OR over the ranks, into every rank's X
        const int64_t wi = (reinterpret_cast<float*>(xmask) - a.x) + 4 * p + lane;
        uint32_t m = 0;
        for (int r = 0; r < N; r++) m |= __ldcv(reinterpret_cast<const unsigned int*>(a.x_peer[r] + wi));
        for (int r = 0; r < N; r++) *reinterpret_cast<uint32_t*>(a.x_peer[r] + wi) = m;
      }
      if (i >= total4) continue;
      if (a.x_mc != nullptr) {
        const float4 v = multimem_ld_reduce4(a.x_mc + 4 * i);
        multimem_st4(a.x_mc + 4 * i, v);
      } else {
        float4 v = f4_zero();
        for (int r0 = 0; r0 < N; r0 += 4) {          // four remote loads in flight, summed in rank order
          float4 t[4];
#pragma unroll
          for (int q = 0; q < 4; q++)
            t[q] = (r0 + q < N) ? ld_cv4(reinterpret_cast<const float4*>(a.x_peer[r0 + q]) + i) : f4_zero();
#pragma unroll
          for (int q = 0; q < 4; q++)
            if (r0 + q < N) v = f4_add(v, t[q]);
        }
        for (int r = 0; r < N; r++) reinterpret_cast<float4*>(a.x_peer[r])[i] = v;
      }
    }
    __syncthreads();
    if (threadIdx.x < 32 && !cross_rank_flags(a, 1, step + 1)) a.state[1] = 1;
    __syncthreads();
    // ---- C: optimizer over my pieces ----
    for (int64_t L = pslot;; L += kSlots) {
      const int64_t p = piece_of(L);
      if (p >= n_pieces) break;
      const int64_t i = p * kPiece + lane;
      if (i >= total4) continue;
      const float4 v = ld_cv4(x4 + i);
      const uint32_t tbits = TOUCHED ? (__ldcv(reinterpret_cast<const unsigned int*>(xmask) + 4 * p + (lane >> 3)) >> (4 * (lane & 7))) & 0xFu
                                     : 0u;
      if (i == n_g4) { loss_all = v.x; has_loss = true; }
      else reg += apply(i, v, tbits);
    }
  }

  // ---- loss: per-CTA regulariser partials, the last CTA to finish adds them up in a fixed order ----
  {
    const float br = block_sum(reg, scratch);
    if (threadIdx.x == 0) a.sq_ws[b] = br;
    if (has_loss) a.sq_ws[G] = loss_all;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(a.state + 2, 1) == G - 1) ? 1 : 0;
    __syncthreads();
    if (s_last && threadIdx.x < 32) {
      __threadfence();
      float r = 0.f;
      for (int i = lane; i < G; i += 32) r += __ldcv(a.sq_ws + i);
      r = warp_sum(r);
      if (lane == 0) {
        a.loss_out[0] = __ldcv(a.sq_ws + G) + r;
        a.state[2] = 0;
        a.state[0] = step + 1;
      }
    }
  }
}

template <int KIND, bool TOUCHED>
static int launch_dp(const DpArgs& a, cudaStream_t st) {
  static int grid_cached = 0;
  if (grid_cached == 0) {
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dp_step_kernel<KIND, TOUCHED>, kDpThreads, 0);
    if (e != cudaSuccess || per_sm < 1) {
      set_error("dp_step: occupancy query failed: %s", cudaGetErrorString(e));
      cudaGetLastError();
      return HHFM_ERR_LAUNCH;
    }
    grid_cached = sm_count();      // one CTA per SM: every CTA is resident, grid.sync() is legal
  }
  // One CTA per SM and at least one resident CTA per SM (checked above): the whole grid is resident as soon as the previous
  // kernel of the stream has drained, which is all the cross-GPU flag waits need (a CTA never waits for a CTA of its own
  // grid).  A cooperative launch would guarantee it formally but costs tens of microseconds per step; HHFM_DP_COOP=1 selects it.
  static const bool coop = [] { const char* e = getenv("HHFM_DP_COOP"); return e && e[0] == '1'; }();
  cudaError_t e = cudaSuccess;
  if (a.n_ranks == 1 || !coop) {
    dp_step_kernel<KIND, TOUCHED><<<grid_cached, kDpThreads, 0, st>>>(a);
  } else {
    void* params[] = {(void*)&a};
    e = cudaLaunchCooperativeKernel((const void*)dp_step_kernel<KIND, TOUCHED>, dim3(grid_cached), dim3(kDpThreads), params, 0, st);
  }
  if (e != cudaSuccess) {
    set_error("dp_step_kernel: cooperative launch failed: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return HHFM_ERR_LAUNCH;
  }
  return check_launch("dp_step_kernel");
}

}  // namespace hhfm

using namespace hhfm;

extern "C" int64_t hhfm_dp_exchange_floats(int64_t n_grad) {
  if (n_grad < 1) return -1;
  return ((n_grad + 3) / 4 + 1) * 4;
}

extern "C" int64_t hhfm_dp_flag_ints(void) { return 2 * 256 * kMaxPeers; }

// argument checks and DpArgs of hhfm_dp_step / hhfm_dp_step_touched (the segments' widths are 0: dense)
static int dp_prepare(DpArgs& a, int32_t kind, const hhfm_dp_segment* segs, int32_t n_segs, float* arena, int64_t n_grad,
                      float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot, int64_t K, int64_t M, const int32_t* hot_slot,
                      int64_t bias_off, const float* loss_partials, float* x_local, float* x_multicast, const int64_t* x_peers_host,
                      const int64_t* flag_peers_host, int32_t rank, int32_t n_ranks, int32_t* state, float lr, float beta1,
                      float beta2, float eps, float* reg_workspace, float* loss_out, double timeout_s) {
  HHFM_REQUIRE(segs && n_segs >= 1 && n_segs <= kMaxSegs, "dp_step: 1..4 segments");
  HHFM_REQUIRE(arena && n_grad > 0 && loss_partials && x_local && state && reg_workspace && loss_out, "dp_step: NULL argument");
  HHFM_REQUIRE(n_ranks >= 1 && n_ranks <= kMaxPeers && rank >= 0 && rank < n_ranks, "dp_step: bad rank / n_ranks");
  HHFM_REQUIRE(n_ranks == 1 || (x_peers_host && flag_peers_host), "dp_step: peer tables required for n_ranks > 1");
  HHFM_REQUIRE(sm_count() <= 256, "dp_step: the flag arrays are sized for at most 256 CTAs");
  HHFM_REQUIRE((((uintptr_t)arena | (uintptr_t)x_local | (uintptr_t)x_multicast) & 15) == 0, "dp_step: buffers must be 16-byte aligned");
  HHFM_REQUIRE(K > 0 && K % 4 == 0 && M > 0 && M * K <= n_grad, "dp_step: the table gradient [M, K] must lead the arena");
  HHFM_REQUIRE(ghot == nullptr || (n_rep >= 1 && n_hot >= 1 && hot_slot), "dp_step: bad hot-row plan");
  HHFM_REQUIRE(kind >= HHFM_OPT_ADAGRAD && kind <= HHFM_OPT_SGD, "dp_step: unknown optimizer kind %d", kind);
  memset(&a, 0, sizeof(a));
  a.n_seg = n_segs;
  for (int i = 0; i < n_segs; i++) {
    const hhfm_dp_segment& s = segs[i];
    HHFM_REQUIRE(s.w && s.n > 0 && s.offset >= 0 && s.offset + s.n <= n_grad, "dp_step: segment outside the gradient range");
    HHFM_REQUIRE(kind == HHFM_OPT_SGD || s.s1, "dp_step: optimizer state is NULL");
    HHFM_REQUIRE(kind != HHFM_OPT_ADAM || s.s2, "dp_step: adam needs two state buffers");
    HHFM_REQUIRE((s.offset & 3) != 0 || s.n < 4 || (((uintptr_t)s.w | (uintptr_t)s.s1 | (uintptr_t)s.s2) & 15) == 0,
                 "dp_step: segment buffers must be 16-byte aligned");
    a.seg[i] = DpSeg{s.w, s.s1, s.s2, s.offset, s.n, s.lamda, 0};
  }
  a.arena = arena;
  a.n_g = n_grad;
  a.ghot = (ghot && n_hot > 0) ? ghot : nullptr;
  a.ghot_bias = a.ghot ? ghot_bias : nullptr;
  a.n_rep = n_rep;
  a.n_hot = n_hot;
  a.K = (int)K;
  a.hot_slot = hot_slot;
  a.M = M;
  a.bias_off = bias_off;
  HHFM_REQUIRE(a.ghot_bias == nullptr || bias_off >= 0, "dp_step: bias_off required with ghot_bias");
  a.loss_partials = loss_partials;
  a.x = x_local;
  a.x_mc = (n_ranks > 1) ? x_multicast : nullptr;
  for (int r = 0; r < n_ranks && n_ranks > 1; r++) {
    a.x_peer[r] = reinterpret_cast<float*>(x_peers_host[r]);
    a.flag_peer[r] = reinterpret_cast<int32_t*>(flag_peers_host[r]);
    HHFM_REQUIRE(a.x_peer[r] && a.flag_peer[r] && ((uintptr_t)a.x_peer[r] & 15) == 0, "dp_step: bad peer address");
  }
  a.rank = rank;
  a.n_ranks = n_ranks;
  a.state = state;
  a.p = OptP2{lr, 0.f, beta1, beta2, eps};
  a.sq_ws = reg_workspace;
  a.loss_out = loss_out;
  if (timeout_s <= 0) timeout_s = 120.0;
  a.timeout_cycles = (long long)(timeout_s * 1.9e9);
  {
    // Off by default: `st.release.sys` after the CTA barrier is cumulative over the CTA's stores and `ld.acquire.sys` before
    // the next CTA barrier orders the CTA's loads; the explicit membar.sys pairs cost 13 us per step at N = 2 (0.738 -> 0.725 ms)
    static const int fences = [] { const char* e = getenv("HHFM_DP_FENCES"); return (e && e[0] == '1') ? 1 : 0; }();
    a.fences = fences;
  }
  return HHFM_OK;
}

template <bool TOUCHED>
static int launch_dp_kind(int32_t kind, const DpArgs& a, cudaStream_t st) {
  switch (kind) {
    case HHFM_OPT_ADAGRAD: return launch_dp<HHFM_OPT_ADAGRAD, TOUCHED>(a, st);
    case HHFM_OPT_ADAM: return launch_dp<HHFM_OPT_ADAM, TOUCHED>(a, st);
    case HHFM_OPT_MOMENTUM: return launch_dp<HHFM_OPT_MOMENTUM, TOUCHED>(a, st);
    case HHFM_OPT_SGD: return launch_dp<HHFM_OPT_SGD, TOUCHED>(a, st);
    default: set_error("dp_step: unknown optimizer kind %d", kind); return HHFM_ERR_BAD_ARG;
  }
}

extern "C" int hhfm_dp_step(int32_t kind, const hhfm_dp_segment* segs, int32_t n_segs, float* arena, int64_t n_grad,
                            float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot, int64_t K, int64_t M,
                            const int32_t* hot_slot, int64_t bias_off, const float* loss_partials, float* x_local, float* x_multicast,
                            const int64_t* x_peers_host, const int64_t* flag_peers_host, int32_t rank, int32_t n_ranks,
                            int32_t* state, float lr, float beta1, float beta2, float eps, float* reg_workspace,
                            float* loss_out, double timeout_s, hhfm_stream_t stream) {
  DpArgs a;
  const int rc = dp_prepare(a, kind, segs, n_segs, arena, n_grad, ghot, ghot_bias, n_rep, n_hot, K, M, hot_slot, bias_off,
                            loss_partials, x_local, x_multicast, x_peers_host, flag_peers_host, rank, n_ranks, state, lr, beta1,
                            beta2, eps, reg_workspace, loss_out, timeout_s);
  if (rc != HHFM_OK) return rc;
  return launch_dp_kind<false>(kind, a, (cudaStream_t)stream);
}

extern "C" int64_t hhfm_dp_exchange_floats_touched(int64_t n_grad) {
  if (n_grad < 1) return -1;
  const int64_t total4 = (n_grad + 3) / 4 + 1;
  return (total4 + (total4 + kPiece - 1) / kPiece) * 4;
}

extern "C" int hhfm_dp_step_touched(int32_t kind, const hhfm_dp_segment* segs, int32_t n_segs, const int32_t* seg_widths,
                                    const int32_t* stamps, int32_t stamp, float* arena, int64_t n_grad, float* ghot,
                                    float* ghot_bias, int32_t n_rep, int32_t n_hot, int64_t K, int64_t M,
                                    const int32_t* hot_slot, int64_t bias_off, const float* loss_partials, float* x_local,
                                    float* x_multicast, const int64_t* x_peers_host, const int64_t* flag_peers_host,
                                    int32_t rank, int32_t n_ranks, int32_t* state, float lr, float beta1, float beta2,
                                    float eps, float* reg_workspace, float* loss_out, double timeout_s, hhfm_stream_t stream) {
  HHFM_REQUIRE(seg_widths, "dp_step_touched: seg_widths is NULL");
  DpArgs a;
  const int rc = dp_prepare(a, kind, segs, n_segs, arena, n_grad, ghot, ghot_bias, n_rep, n_hot, K, M, hot_slot, bias_off,
                            loss_partials, x_local, x_multicast, x_peers_host, flag_peers_host, rank, n_ranks, state, lr, beta1,
                            beta2, eps, reg_workspace, loss_out, timeout_s);
  if (rc != HHFM_OK) return rc;
  for (int i = 0; i < n_segs; i++) {
    const int32_t wd = seg_widths[i];
    HHFM_REQUIRE(wd >= 0, "dp_step_touched: negative row width");
    if (wd == 0) continue;
    HHFM_REQUIRE(stamps, "dp_step_touched: a segment with a row width needs the stamp array");
    HHFM_REQUIRE(segs[i].n % wd == 0 && segs[i].n / wd <= M, "dp_step_touched: segment %d is not [rows <= M, width]", i);
    HHFM_REQUIRE(segs[i].lamda == 0.f, "dp_step_touched: a segment with a row width takes no L2 term");
    a.seg[i].width = wd;
  }
  a.stamps = stamps;
  a.stamp = stamp;
  return launch_dp_kind<true>(kind, a, (cudaStream_t)stream);
}
