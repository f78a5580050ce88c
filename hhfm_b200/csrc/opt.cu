// K4 generic row scatter-add, K5 TF-1.x optimizers (dense-with-L2 and touched-rows variants), loss finalize.
// Reference: tf.train.{Adagrad,Adam,Momentum,GradientDescent}Optimizer.minimize (FM.py:129-136, BPR.py:93,
// MF.py:104).  TF kernels restated: ApplyAdagrad `accum += g*g; var -= lr*g*rsqrt(accum)` (no epsilon),
// ApplyAdam with lr_t folded by the caller, ApplyMomentum `accum = accum*mu + g; var -= lr*accum`.
// All kernels are pure streaming float4 passes (HBM-bound): read g,w,state -> write w,state,(g=0).
#include "common.cuh"
#include "staged.cuh"

namespace hhfm {

struct OptP {
  float lr, lamda, p1, p2, p3;   // adam: p1=beta1 p2=beta2 p3=eps ; momentum: p1=mu
};

template <int KIND>
__device__ __forceinline__ void opt_elem(float& w, float& s1, float& s2, float g, const OptP& p) {
  if (KIND == HHFM_OPT_ADAGRAD) {
    s1 = fmaf(g, g, s1);                                // explicit contractions: the same bits as p2p.cu::opt_elem2
    w = w - p.lr * g / sqrtf(s1);
  } else if (KIND == HHFM_OPT_ADAM) {
    s1 = fmaf(p.p1, s1, (1.f - p.p1) * g);
    s2 = fmaf(p.p2, s2, (1.f - p.p2) * (g * g));
    w = w - p.lr * s1 / (sqrtf(s2) + p.p3);
  } else if (KIND == HHFM_OPT_MOMENTUM) {
    s1 = fmaf(s1, p.p1, g);
    w = fmaf(-p.lr, s1, w);
  } else {
    w = fmaf(-p.lr, g, w);
  }
}

template <int KIND>
__device__ __forceinline__ void opt_vec4(float4& w, float4& s1, float4& s2, float4 g, const OptP& p) {
  opt_elem<KIND>(w.x, s1.x, s2.x, g.x, p);
  opt_elem<KIND>(w.y, s1.y, s2.y, g.y, p);
  opt_elem<KIND>(w.z, s1.z, s2.z, g.z, p);
  opt_elem<KIND>(w.w, s1.w, s2.w, g.w, p);
}

// dense: n elements, g_eff = g + lamda*w.  Handles n % 4 != 0 with a scalar tail (bias vectors, scalars).
template <int KIND>
__global__ void __launch_bounds__(256) opt_dense_kernel(float* __restrict__ w, float* __restrict__ s1,
                                                        float* __restrict__ s2, float* __restrict__ g, int64_t n,
                                                        OptP p, int zero_grad, float* sq_partials) {
  __shared__ float scratch[32];
  const int64_t n4 = n >> 2;
  float sq = 0.f;
  float4* w4 = reinterpret_cast<float4*>(w);
  float4* g4 = reinterpret_cast<float4*>(g);
  float4* a4 = reinterpret_cast<float4*>(s1);
  float4* b4 = reinterpret_cast<float4*>(s2);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 wv = w4[i], gv = g4[i];
    float4 av = (KIND != HHFM_OPT_SGD) ? a4[i] : f4_zero();
    float4 bv = (KIND == HHFM_OPT_ADAM) ? b4[i] : f4_zero();
    sq += f4_dot(wv, wv);
    gv = f4_fma(wv, p.lamda, gv);
    opt_vec4<KIND>(wv, av, bv, gv, p);
    w4[i] = wv;
    if (KIND != HHFM_OPT_SGD) a4[i] = av;
    if (KIND == HHFM_OPT_ADAM) b4[i] = bv;
    if (zero_grad) g4[i] = f4_zero();
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    float wv = w[i], gv = g[i];
    float av = (KIND != HHFM_OPT_SGD) ? s1[i] : 0.f;
    float bv = (KIND == HHFM_OPT_ADAM) ? s2[i] : 0.f;
    sq += wv * wv;
    gv = fmaf(wv, p.lamda, gv);
    opt_elem<KIND>(wv, av, bv, gv, p);
    w[i] = wv;
    if (KIND != HHFM_OPT_SGD) s1[i] = av;
    if (KIND == HHFM_OPT_ADAM) s2[i] = bv;
    if (zero_grad) g[i] = 0.f;
  }
  if (sq_partials != nullptr) {
    const float b = block_sum(sq, scratch);
    write_partial(sq_partials, b);
  }
}

// rows: only rows[0 .. *n_rows) move (TF SparseApply*), K elements each; K % 4 == 0 or K == 1.
template <int KIND>
__global__ void __launch_bounds__(256) opt_rows_kernel(float* __restrict__ w, float* __restrict__ s1,
                                                       float* __restrict__ g, const int32_t* __restrict__ rows,
                                                       const int32_t* __restrict__ n_rows_dev, int K, OptP p,
                                                       int zero_grad) {
  const int n_rows = *n_rows_dev;
  float dummy = 0.f;
  if (K == 1) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (int64_t)gridDim.x * blockDim.x) {
      const int r = rows[i];
      float wv = w[r], gv = g[r], av = (KIND != HHFM_OPT_SGD) ? s1[r] : 0.f;
      opt_elem<KIND>(wv, av, dummy, gv, p);
      w[r] = wv;
      if (KIND != HHFM_OPT_SGD) s1[r] = av;
      if (zero_grad) g[r] = 0.f;
    }
    return;
  }
  const int kv = K >> 2;
  const int64_t total = (int64_t)n_rows * kv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = rows[i / kv];
    const int64_t off = (int64_t)r * kv + (i % kv);
    float4 wv = reinterpret_cast<float4*>(w)[off], gv = reinterpret_cast<float4*>(g)[off];
    float4 av = (KIND != HHFM_OPT_SGD) ? reinterpret_cast<float4*>(s1)[off] : f4_zero();
    float4 bv = f4_zero();
    opt_vec4<KIND>(wv, av, bv, gv, p);
    reinterpret_cast<float4*>(w)[off] = wv;
    if (KIND != HHFM_OPT_SGD) reinterpret_cast<float4*>(s1)[off] = av;
    if (zero_grad) reinterpret_cast<float4*>(g)[off] = f4_zero();
  }
}

__global__ void __launch_bounds__(256) scatter_rows_kernel(const int32_t* __restrict__ rows, const float* __restrict__ src,
                                                           int64_t n, int K, float* __restrict__ dst) {
  const int kv = K >> 2;
  const int64_t total = n * kv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / kv;
    const int c = (int)(i % kv);
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    red_add_v4(dst + (size_t)__ldg(rows + r) * K + 4 * c, v);
  }
}

__global__ void scatter_scalar_kernel(const int32_t* __restrict__ rows, const float* __restrict__ src, int64_t n,
                                      float* __restrict__ dst) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    atomicAdd(dst + __ldg(rows + i), __ldg(src + i));
}

// Fold the n_rep replicas of the hot-row accumulators into the gradient table (fixed order: deterministic) and
// clear them for the next step.  One thread per float4 of a hot row (+ one per bias slot).
__global__ void __launch_bounds__(256) hot_fold_kernel(float* __restrict__ ghot, float* __restrict__ ghot_bias, int n_rep,
                                                       int n_hot, int K, const int32_t* __restrict__ hot_rows,
                                                       float* __restrict__ gV, float* __restrict__ gbias) {
  const int kv = K >> 2;
  const int64_t total = (int64_t)n_hot * kv;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) {
    const int s = (int)(i / kv), c = (int)(i % kv);
    float4 acc = f4_zero();
    // eight replica loads in flight per thread (the plain loop was a chain of n_rep dependent L2 round trips); the sum is
    // still formed in replica order, so it is reproducible
    for (int r0 = 0; r0 < n_rep; r0 += 8) {
      float4 t[8];
#pragma unroll
      for (int q = 0; q < 8; q++) {
        float4* p = reinterpret_cast<float4*>(ghot + ((size_t)(r0 + q) * n_hot + s) * K) + c;
        t[q] = (r0 + q < n_rep) ? *p : f4_zero();
      }
#pragma unroll
      for (int q = 0; q < 8; q++) {
        if (r0 + q < n_rep) {
          acc = f4_add(acc, t[q]);
          *(reinterpret_cast<float4*>(ghot + ((size_t)(r0 + q) * n_hot + s) * K) + c) = f4_zero();
        }
      }
    }
    float4* d = reinterpret_cast<float4*>(gV + (size_t)hot_rows[s] * K) + c;
    *d = f4_add(*d, acc);
  } else if (ghot_bias != nullptr && gbias != nullptr && i < total + n_hot) {
    const int s = (int)(i - total);
    float acc = 0.f;
    for (int r = 0; r < n_rep; r++) {
      float* p = ghot_bias + (size_t)r * n_hot + s;
      acc += *p;
      *p = 0.f;
    }
    gbias[hot_rows[s]] += acc;
  }
}

// loss = sum(loss_partials) + half_lamda * sum(sq_partials): one warp, fixed order -> deterministic.
__global__ void loss_finalize_kernel(const float* __restrict__ lp, const float* __restrict__ sp, float half_lamda,
                                     float* __restrict__ out) {
  float a = 0.f, b = 0.f;
  for (int i = threadIdx.x; i < kPartials; i += 32) {
    a += lp[i];
    if (sp) b += sp[i];
  }
  a = warp_sum(a);
  b = warp_sum(b);
  if (threadIdx.x == 0) out[0] = a + half_lamda * b;
}

static int dense_grid(int64_t n) {
  int64_t need = ((n >> 2) + 255) / 256;
  int64_t cap = (int64_t)sm_count() * 8;
  if (cap > kPartials) cap = kPartials;
  if (need < 1) need = 1;
  return (int)(need < cap ? need : cap);
}

template <int KIND>
static int launch_dense(float* w, float* s1, float* s2, float* g, int64_t n, OptP p, int zero_grad, float* sq_partials,
                        cudaStream_t st) {
  HHFM_REQUIRE(w && g && n > 0, "opt_dense: w, g required and n > 0");
  HHFM_REQUIRE(KIND == HHFM_OPT_SGD || s1, "opt_dense: optimizer state is NULL");
  HHFM_REQUIRE(KIND != HHFM_OPT_ADAM || s2, "opt_dense: adam needs two state buffers");
  HHFM_REQUIRE((((uintptr_t)w | (uintptr_t)g | (uintptr_t)s1 | (uintptr_t)s2) & 15) == 0 || n < 4,
               "opt_dense: buffers must be 16-byte aligned");
  opt_dense_kernel<KIND><<<dense_grid(n), 256, 0, st>>>(w, s1, s2, g, n, p, zero_grad, sq_partials);
  return check_launch("opt_dense_kernel");
}

template <int KIND>
static int launch_rows(float* w, float* s1, float* g, const int32_t* rows, const int32_t* n_rows_dev, int64_t max_rows,
                       int64_t K, OptP p, int zero_grad, cudaStream_t st) {
  HHFM_REQUIRE(w && g && rows && n_rows_dev, "opt_rows: w, g, rows, n_rows_dev required");
  HHFM_REQUIRE(KIND == HHFM_OPT_SGD || s1, "opt_rows: optimizer state is NULL");
  HHFM_REQUIRE(K == 1 || (K % 4 == 0 && K > 0), "opt_rows: K must be 1 or a multiple of 4");
  HHFM_REQUIRE(max_rows > 0, "opt_rows: max_rows must be > 0");
  int64_t work = K == 1 ? max_rows : max_rows * (K >> 2);
  int64_t need = (work + 255) / 256;
  int64_t cap = (int64_t)sm_count() * 8;
  int grid = (int)(need < cap ? need : cap);
  if (grid < 1) grid = 1;
  opt_rows_kernel<KIND><<<grid, 256, 0, st>>>(w, s1, g, rows, n_rows_dev, (int)K, p, zero_grad);
  return check_launch("opt_rows_kernel");
}

// ---- coalesced-sparse gradient exchange (SURVEY 8e): pack the touched rows of a dense gradient, mark received rows ----
__global__ void __launch_bounds__(256) gather_rows_kernel(float* __restrict__ table, const int32_t* __restrict__ ids, int64_t n, int K,
                                                          float* __restrict__ out, int zero_src) {
  if (K == 1) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      const int r = __ldg(ids + i);
      out[i] = table[r];
      if (zero_src) table[r] = 0.f;
    }
    return;
  }
  const int kv = K >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * kv; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / kv;
    const int c = (int)(i % kv);
    float4* src = reinterpret_cast<float4*>(table) + (size_t)__ldg(ids + row) * kv + c;
    reinterpret_cast<float4*>(out)[i] = *src;
    if (zero_src) *src = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

__global__ void __launch_bounds__(256) touch_rows_kernel(const int32_t* __restrict__ ids, int64_t n, int32_t* stamp_arr, int32_t stamp,
                                                         int32_t* rows, int32_t* count) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    touch_row(stamp_arr, stamp, rows, count, __ldg(ids + i));
}

// plain stamp stores (padding ids < 0 skipped); the list is produced by launch_touched_compact afterwards
__global__ void __launch_bounds__(256) mark_rows_kernel(const int32_t* __restrict__ ids, int64_t n, int32_t* __restrict__ stamp_arr,
                                                        int32_t stamp) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int id = __ldg(ids + i);
    if (id >= 0) stamp_arr[id] = stamp;
  }
}

// Lazy-exact dense L2 (SURVEY.md 7, hard part 2-ii).  The reference's l2_regularizer on the table (FM.py:124,
// OurModel7.py:181-182) makes every row move every step: g = lamda*w; acc += g^2; w -= lr*g/sqrt(acc).  For a row that no
// sample touches those steps depend on nothing but the row itself, so they can be replayed later, element by element, with
// the same fp32 operations in the same order: bit-identical to the dense kernel.  `last_step[row]` = the last optimizer step
// the row reflects; this kernel replays steps last+1 .. upto for the listed rows (rows == NULL: all M rows).
__global__ void __launch_bounds__(256) adagrad_l2_replay_kernel(float* __restrict__ w, float* __restrict__ acc,
                                                                int32_t* __restrict__ last_step, const int32_t* __restrict__ rows,
                                                                const int32_t* __restrict__ n_rows_dev, int64_t M, int K, OptP p,
                                                                int32_t upto) {
  const int kv = K >> 2;
  const int64_t n_rows = rows ? (int64_t)*n_rows_dev : M;
  const int64_t total = n_rows * kv;
  float dummy = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t li = i / kv;
    const int r = rows ? rows[li] : (int)li;
    const int n = upto - last_step[r];
    if (n > 0) {
      const int64_t off = (int64_t)r * kv + (i % kv);
      float4 wv = reinterpret_cast<float4*>(w)[off], av = reinterpret_cast<float4*>(acc)[off];
      for (int s = 0; s < n; s++) {
        opt_elem<HHFM_OPT_ADAGRAD>(wv.x, av.x, dummy, fmaf(wv.x, p.lamda, 0.f), p);
        opt_elem<HHFM_OPT_ADAGRAD>(wv.y, av.y, dummy, fmaf(wv.y, p.lamda, 0.f), p);
        opt_elem<HHFM_OPT_ADAGRAD>(wv.z, av.z, dummy, fmaf(wv.z, p.lamda, 0.f), p);
        opt_elem<HHFM_OPT_ADAGRAD>(wv.w, av.w, dummy, fmaf(wv.w, p.lamda, 0.f), p);
      }
      reinterpret_cast<float4*>(w)[off] = wv;
      reinterpret_cast<float4*>(acc)[off] = av;
    }
  }
}

// every chunk of a row reads last_step before any chunk of that row may overwrite it: the stamps are written by a second
// launch
__global__ void __launch_bounds__(256) set_last_step_kernel(int32_t* __restrict__ last_step, const int32_t* __restrict__ rows,
                                                            const int32_t* __restrict__ n_rows_dev, int64_t M, int32_t value) {
  const int64_t n_rows = rows ? (int64_t)*n_rows_dev : M;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (int64_t)gridDim.x * blockDim.x)
    last_step[rows ? rows[i] : i] = value;
}

// SparseApplyAdagrad on the listed rows with the dense L2 term of this step: g_eff = g + lamda*w (same expression as
// opt_dense_kernel); the caller stamps last_step = t afterwards.
__global__ void __launch_bounds__(256) adagrad_rows_l2_kernel(float* __restrict__ w, float* __restrict__ acc, float* __restrict__ g,
                                                              const int32_t* __restrict__ rows, const int32_t* __restrict__ n_rows_dev,
                                                              int K, OptP p, int zero_grad) {
  const int n_rows = *n_rows_dev;
  const int kv = K >> 2;
  const int64_t total = (int64_t)n_rows * kv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = rows[i / kv];
    const int64_t off = (int64_t)r * kv + (i % kv);
    float4 wv = reinterpret_cast<float4*>(w)[off], gv = reinterpret_cast<float4*>(g)[off];
    float4 av = reinterpret_cast<float4*>(acc)[off];
    float4 bv = f4_zero();
    gv = f4_fma(wv, p.lamda, gv);
    opt_vec4<HHFM_OPT_ADAGRAD>(wv, av, bv, gv, p);
    reinterpret_cast<float4*>(w)[off] = wv;
    reinterpret_cast<float4*>(acc)[off] = av;
    if (zero_grad) reinterpret_cast<float4*>(g)[off] = f4_zero();
  }
}

// Measurement aid (bench.py `roofline.peak` of the L2-bound kernels): every thread streams the whole buffer `iters` times
// with 16-byte loads that bypass L1 (ld.global.cg), so a buffer that fits the 126 MB L2 is served by L2 only.
__global__ void __launch_bounds__(256) l2_read_sweep_kernel(const float4* __restrict__ buf, int64_t n4, int iters, float* sink) {
  float4 acc = f4_zero();
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  for (int it = 0; it < iters; it++) {
    int64_t i = tid;
    for (; i + 3 * nth < n4; i += 4 * nth) {
      const float4 a = __ldcg(buf + i), b = __ldcg(buf + i + nth), c = __ldcg(buf + i + 2 * nth), d = __ldcg(buf + i + 3 * nth);
      acc = f4_add(acc, f4_add(f4_add(a, b), f4_add(c, d)));
    }
    for (; i < n4; i += nth) acc = f4_add(acc, __ldcg(buf + i));
  }
  if (f4_hsum(acc) == 123.456f) *sink = 1.f;      // keeps the loads alive without a store on the hot path
}

}  // namespace hhfm

using namespace hhfm;

extern "C" int hhfm_l2_read_sweep(const float* buf, int64_t n_floats, int32_t iters, float* sink, hhfm_stream_t stream) {
  HHFM_REQUIRE(buf && sink && n_floats >= 4 && iters >= 1 && ((uintptr_t)buf & 15) == 0, "l2_read_sweep: bad arguments");
  l2_read_sweep_kernel<<<sm_count() * 8, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(buf), n_floats >> 2, iters, sink);
  return check_launch("l2_read_sweep_kernel");
}

extern "C" int hhfm_opt_adagrad_dense_l2(float* w, float* acc, float* g, int64_t n, float lr, float lamda,
                                         int32_t zero_grad, float* sq_partials, hhfm_stream_t stream) {
  OptP p{lr, lamda, 0.f, 0.f, 0.f};
  return launch_dense<HHFM_OPT_ADAGRAD>(w, acc, nullptr, g, n, p, zero_grad, sq_partials, (cudaStream_t)stream);
}
extern "C" int hhfm_opt_adam_dense_l2(float* w, float* m, float* v, float* g, int64_t n, float lr_t, float beta1,
                                      float beta2, float eps, float lamda, int32_t zero_grad, float* sq_partials,
                                      hhfm_stream_t stream) {
  OptP p{lr_t, lamda, beta1, beta2, eps};
  return launch_dense<HHFM_OPT_ADAM>(w, m, v, g, n, p, zero_grad, sq_partials, (cudaStream_t)stream);
}
extern "C" int hhfm_opt_momentum_dense_l2(float* w, float* acc, float* g, int64_t n, float lr, float momentum,
                                          float lamda, int32_t zero_grad, float* sq_partials, hhfm_stream_t stream) {
  OptP p{lr, lamda, momentum, 0.f, 0.f};
  return launch_dense<HHFM_OPT_MOMENTUM>(w, acc, nullptr, g, n, p, zero_grad, sq_partials, (cudaStream_t)stream);
}
extern "C" int hhfm_opt_sgd_dense_l2(float* w, float* g, int64_t n, float lr, float lamda, int32_t zero_grad,
                                     float* sq_partials, hhfm_stream_t stream) {
  OptP p{lr, lamda, 0.f, 0.f, 0.f};
  return launch_dense<HHFM_OPT_SGD>(w, nullptr, nullptr, g, n, p, zero_grad, sq_partials, (cudaStream_t)stream);
}
extern "C" int hhfm_opt_adagrad_rows(float* w, float* acc, float* g, const int32_t* rows, const int32_t* n_rows_dev,
                                     int64_t max_rows, int64_t K, float lr, int32_t zero_grad, hhfm_stream_t stream) {
  OptP p{lr, 0.f, 0.f, 0.f, 0.f};
  return launch_rows<HHFM_OPT_ADAGRAD>(w, acc, g, rows, n_rows_dev, max_rows, K, p, zero_grad, (cudaStream_t)stream);
}
extern "C" int hhfm_opt_momentum_rows(float* w, float* acc, float* g, const int32_t* rows, const int32_t* n_rows_dev,
                                      int64_t max_rows, int64_t K, float lr, float momentum, int32_t zero_grad,
                                      hhfm_stream_t stream) {
  OptP p{lr, 0.f, momentum, 0.f, 0.f};
  return launch_rows<HHFM_OPT_MOMENTUM>(w, acc, g, rows, n_rows_dev, max_rows, K, p, zero_grad, (cudaStream_t)stream);
}
extern "C" int hhfm_opt_sgd_rows(float* w, float* g, const int32_t* rows, const int32_t* n_rows_dev, int64_t max_rows,
                                 int64_t K, float lr, int32_t zero_grad, hhfm_stream_t stream) {
  OptP p{lr, 0.f, 0.f, 0.f, 0.f};
  return launch_rows<HHFM_OPT_SGD>(w, nullptr, g, rows, n_rows_dev, max_rows, K, p, zero_grad, (cudaStream_t)stream);
}

extern "C" int hhfm_scatter_add_rows(const int32_t* rows, const float* src, int64_t n, int64_t K, float* dst, int64_t M,
                                     hhfm_stream_t stream) {
  HHFM_REQUIRE(rows && src && dst && M > 0, "scatter_add_rows: NULL argument");
  HHFM_REQUIRE(K == 1 || (K > 0 && K % 4 == 0), "scatter_add_rows: K must be 1 or a multiple of 4");
  if (n == 0) return HHFM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t work = K == 1 ? n : n * (K >> 2);
  int64_t need = (work + 255) / 256, cap = (int64_t)sm_count() * 8;
  int grid = (int)(need < cap ? need : cap);
  if (K == 1) scatter_scalar_kernel<<<grid, 256, 0, st>>>(rows, src, n, dst);
  else scatter_rows_kernel<<<grid, 256, 0, st>>>(rows, src, n, (int)K, dst);
  return check_launch("scatter_rows_kernel");
}

extern "C" int hhfm_hot_fold(float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot, int64_t K,
                             const int32_t* hot_rows, float* gV, float* gbias, hhfm_stream_t stream) {
  HHFM_REQUIRE(ghot && hot_rows && gV, "hot_fold: NULL argument");
  HHFM_REQUIRE(n_rep >= 1 && n_hot >= 1 && K > 0 && K % 4 == 0, "hot_fold: bad sizes");
  const int64_t total = (int64_t)n_hot * (K >> 2) + n_hot;
  hot_fold_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ghot, ghot_bias, n_rep, n_hot, (int)K,
                                                                                    hot_rows, gV, gbias);
  return check_launch("hot_fold_kernel");
}

extern "C" int hhfm_loss_finalize(const float* loss_partials, const float* sq_partials, float half_lamda, float* loss_out,
                                  hhfm_stream_t stream) {
  HHFM_REQUIRE(loss_partials && loss_out, "loss_finalize: NULL argument");
  loss_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(loss_partials, sq_partials, half_lamda, loss_out);
  return check_launch("loss_finalize_kernel");
}

extern "C" int hhfm_gather_rows(float* table, const int32_t* ids, int64_t n, int64_t K, int64_t M, float* out, int32_t zero_src,
                                hhfm_stream_t stream) {
  HHFM_REQUIRE(table && ids && out && M > 0 && n >= 0, "gather_rows: bad argument");
  HHFM_REQUIRE(K == 1 || (K > 0 && K % 4 == 0), "gather_rows: K must be 1 or a multiple of 4");
  if (n == 0) return HHFM_OK;
  const int64_t work = K == 1 ? n : n * (K >> 2);
  const int64_t need = (work + 255) / 256, cap = (int64_t)sm_count() * 8;
  gather_rows_kernel<<<(int)(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>(table, ids, n, (int)K, out, zero_src);
  return check_launch("gather_rows_kernel");
}

extern "C" int hhfm_mark_rows(const int32_t* ids, int64_t n, int32_t* stamp_arr, int32_t stamp, int64_t M, int32_t* rows,
                              int32_t* count, hhfm_stream_t stream) {
  HHFM_REQUIRE(ids && stamp_arr && rows && count && n >= 0 && M > 0, "mark_rows: bad argument");
  if (n == 0) return HHFM_OK;
  const int64_t need = (n + 255) / 256, cap = (int64_t)sm_count() * 8;
  mark_rows_kernel<<<(int)(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>(ids, n, stamp_arr, stamp);
  int rc = check_launch("mark_rows_kernel");
  if (rc != HHFM_OK) return rc;
  return launch_touched_compact(stamp_arr, stamp, M, rows, count, (cudaStream_t)stream);
}

extern "C" int hhfm_opt_adagrad_l2_replay(float* w, float* acc, int32_t* last_step, const int32_t* rows, const int32_t* n_rows_dev,
                                          int64_t max_rows, int64_t M, int64_t K, float lr, float lamda, int32_t upto,
                                          hhfm_stream_t stream) {
  HHFM_REQUIRE(w && acc && last_step && M > 0 && K > 0 && K % 4 == 0, "opt_adagrad_l2_replay: bad argument");
  HHFM_REQUIRE(!rows || (n_rows_dev && max_rows > 0), "opt_adagrad_l2_replay: rows needs n_rows_dev and max_rows");
  OptP p{lr, lamda, 0.f, 0.f, 0.f};
  const int64_t n = rows ? max_rows : M;
  const int64_t need = (n * (K >> 2) + 255) / 256, cap = (int64_t)sm_count() * 8;
  const int grid = (int)(need < cap ? need : cap);
  cudaStream_t st = (cudaStream_t)stream;
  adagrad_l2_replay_kernel<<<grid, 256, 0, st>>>(w, acc, last_step, rows, n_rows_dev, M, (int)K, p, upto);
  int rc = check_launch("adagrad_l2_replay_kernel");
  if (rc != HHFM_OK) return rc;
  set_last_step_kernel<<<grid, 256, 0, st>>>(last_step, rows, n_rows_dev, M, upto);
  return check_launch("set_last_step_kernel");
}

extern "C" int hhfm_opt_adagrad_rows_l2(float* w, float* acc, float* g, const int32_t* rows, const int32_t* n_rows_dev,
                                        int64_t max_rows, int64_t K, float lr, float lamda, int32_t zero_grad,
                                        int32_t* last_step, int32_t step, hhfm_stream_t stream) {
  HHFM_REQUIRE(w && acc && g && rows && n_rows_dev && last_step && max_rows > 0 && K > 0 && K % 4 == 0,
               "opt_adagrad_rows_l2: bad argument");
  OptP p{lr, lamda, 0.f, 0.f, 0.f};
  const int64_t need = (max_rows * (K >> 2) + 255) / 256, cap = (int64_t)sm_count() * 8;
  const int grid = (int)(need < cap ? need : cap);
  cudaStream_t st = (cudaStream_t)stream;
  adagrad_rows_l2_kernel<<<grid, 256, 0, st>>>(w, acc, g, rows, n_rows_dev, (int)K, p, zero_grad);
  int rc = check_launch("adagrad_rows_l2_kernel");
  if (rc != HHFM_OK) return rc;
  set_last_step_kernel<<<grid, 256, 0, st>>>(last_step, rows, n_rows_dev, 0, step);
  return check_launch("set_last_step_kernel");
}

extern "C" int hhfm_touch_rows(const int32_t* ids, int64_t n, int32_t* stamp_arr, int32_t stamp, int32_t* rows, int32_t* count,
                               hhfm_stream_t stream) {
  HHFM_REQUIRE(ids && stamp_arr && rows && count && n >= 0, "touch_rows: bad argument");
  if (n == 0) return HHFM_OK;
  const int64_t need = (n + 255) / 256, cap = (int64_t)sm_count() * 8;
  touch_rows_kernel<<<(int)(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>(ids, n, stamp_arr, stamp, rows, count);
  return check_launch("touch_rows_kernel");
}
