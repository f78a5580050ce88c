// K2 on the 5th-generation tensor cores: the AFM training pass (Newcode/AFM.py:103-148 + autodiff) as ONE kernel.
//
// The three matrix products of a sample -- Z = P W (attention logits), dP = dZ W^T, dW += P^T dZ, 2*P*K*A flops each --
// run on tcgen05 as 3xTF32 split products (fp32-grade accuracy, see dfm_tc.cu); everything around them (pair products,
// relu, softmax over the pairs, the weighted sum, the chain rule, the embedding scatter) runs in the same CTA between
// the MMA phases, so the [pairs, K] tensors never leave shared memory / TMEM.
//
// Tile = 2 samples = 128 operand rows: sample slot ss owns rows [64 ss, 64 ss + P), the rows P..63 of a slot are zero.
// Thread = (row r, column group): warp & 3 is the TMEM lane quarter (rows), warp >> 2 the group of 16 columns (16 warps).
//   P rows      the thread builds its 16 pair products in registers and writes them (x and lo(x)) with tcgen05.st
//               into TMEM -- the A operand of GEMM 1 -- and, transposed, into the K-major tiles PT[k][r] (A operand of GEMM 3)
//   GEMM 1      Z[128, 64]   = P . W          A = P from TMEM,   B = W^T tiles (K-major smem)   -> TMEM columns [0, 64)
//   epilogue 1  Z row from TMEM, relu, logits; every warp then works out the softmax of its sample slot by itself (lane l
//               looks at pairs l and l + 32, warp shuffles only): with u_p = prediction_W . P_p the output is sum_p a_p u_p,
//               d a_p = g u_p and ds_p = g a_p (u_p - sum_q a_q u_q) -- no afm vector, no CTA-wide reductions.
//               dZ = ds * p * relu' -> TMEM (A operand of GEMM 2) and, transposed, the K-major tiles dZT[a][r]
//   GEMM 2      dP[128, 64]  = dZ . W^T       A = dZ from TMEM,  B = W tiles (K-major smem)     -> TMEM columns [64, 128)
//   GEMM 3      D[128, 64]  += [PT ; PT_lo] . (dZT + dZT_lo)^T   K-major operands, reduction over the 128 tile rows; rows
//               0..63 of D hold P^T dZ, rows 64..127 hold P_lo^T dZ                              -> TMEM columns [128, 192)
//   epilogue 2  dP row from TMEM (+ a_p * d afm) -> shared memory; thread = (slot, field, float4): dE_f = sum_j dP_(f,j) * E_j,
//               one vector reduction per 16 bytes into the gradient table (hot-row replicas as in K1 / K3)
// (tf32 operands can only be MN-major in the SWIZZLE_128B_BASE32B layout, which the K-major products cannot share, so the
// transposed operands of dW are separate tiles written by the same threads -- lane = row makes those stores contiguous.)
// dW is read back from TMEM after every tile and added into registers (two-level accumulation: the tensor core adds into
// its accumulator with truncation, see dfm_tc.cu); the threads add their registers into the global gradient once at the end.
// The column sums over the tile rows (d attention_b, d attention_p, d prediction_W) are deferred: one butterfly step per
// tile into 8 registers, issued behind GEMM 2 / 3, finished once at the end of the kernel.
// Pipeline: the embedding rows (+ bias values, hot-row slots) are fetched with cp.async two tiles ahead (three staging
// buffers), the ids three tiles ahead (ring of four); GEMM 1 of tile t+1 is issued before the scatter of tile t, its A
// operand (P of tile t+1 in TMEM) is built behind GEMM 2 / 3 of tile t; GEMM 2 and GEMM 3 complete on separate mbarriers.
// Three CTA-wide barriers per tile; the scatter of tile t and the PT build of tile t+1 are not separated by one.
//
// Shapes covered: K == A == 64, F <= 11 (P <= 55 pairs).  Everything else stays on the fp32 SIMT kernels (afm.cu).
#include <stdlib.h>

#include "afm.cuh"
#include "staged.cuh"
#include "tc_common.cuh"

namespace hhfm {

namespace aft {

constexpr int KD = 64;                 // K == A
constexpr int kRows = 128;             // operand rows per tile (2 sample slots x 64)
constexpr int kSlot = 64;              // rows per sample slot
constexpr int kMaxF = 11;
constexpr int kEP = KD + 4;            // padded row of the staged embeddings (floats)
constexpr uint32_t kTile = kRows * 128;          // bytes of one [128 rows][32 fp32] operand tile
constexpr uint32_t kWTile = KD * 128;            // bytes of one [64 rows][32 fp32] weight tile
constexpr uint32_t kTmemCols = 512;
// TMEM columns: Z | dP | dW | P x | P lo | dZ x | dZ lo
constexpr uint32_t cZ = 0, cDP = 64, cDW = 128, cPX = 192, cPL = 256, cZX = 320, cZL = 384;

// shared-memory map (bytes); operand tiles are 1024-byte aligned
constexpr uint32_t oP = 0;                              // PT tiles [M = 64 x rows + 64 lo rows][32 r] for r blocks 0..3
constexpr uint32_t oZ = oP + 4 * kTile;                 // dZT tiles: x [64 a rows][32 r] for r blocks 0..3, then lo; reused for the dP rows
constexpr uint32_t oWt = oZ + 4 * kTile;                // W^T tiles (rows = a, contiguous k): [x kb0][x kb1][lo kb0][lo kb1]
constexpr uint32_t oWn = oWt + 4 * kWTile;              // W tiles (rows = k, contiguous a)
constexpr uint32_t kEBytes = 2 * kMaxF * kEP * 4;       // staged embedding rows of one tile: float E[2][kMaxF][kEP]
constexpr uint32_t oE = oWn + 4 * kWTile;               // three tiles in flight: scattered, processed, landing
constexpr uint32_t oMisc = oE + 3 * kEBytes;
constexpr uint32_t kMiscBytes = 10240;
constexpr uint32_t kSmemBytes = oMisc + kMiscBytes + 1024;    // + alignment slack

struct Misc {
  float batt[KD], pvec[KD], wpred[KD];
  float gbatt[KD], gp[KD], gwp[KD];
  float s_part[4][kRows];      // logits by column group
  float u_part[2][4][kRows];   // [tile parity] prediction_W . P_p by column group (built one tile ahead)
  float g[2], bsum[2];
  float biasv[3][2][kMaxF + 1];   // [buffer][slot][field] feature_bias values of the staged rows
  int hslot[3][2][kMaxF + 1];     // [buffer][slot][field] hot-row slot of the staged rows (-1: none)
  int ids[4][2][kMaxF + 1];       // [ring slot][slot][field]: four deep, so the ids of tile t+2 never land on a slot a scatter still reads
  unsigned char pi[kSlot], pj[kSlot];
  unsigned char pidx[kMaxF][kMaxF + 1];
  uint64_t bar1, bar2, bar3;    // GEMM 1 | GEMM 2 | GEMM 3 complete
  uint32_t tmem;
  uint32_t abits[2][2][2];        // DROP: [tile parity][slot][pair / 32] attention-dropout keep bits
  float nvec[2][2][KD];           // DROP: [tile parity][slot][column] pooled-vector dropout factors n_k (0 or 1 / keep)
};
static_assert(sizeof(Misc) <= kMiscBytes, "Misc does not fit its shared-memory slot");

// byte offset of 16-byte chunk c (0..7) of row r inside a 128-byte-swizzled tile
__device__ __forceinline__ uint32_t swz(int r, int c) { return (uint32_t)r * 128u + (uint32_t)((c ^ (r & 7)) << 4); }

// byte offset of fp32 element e (0..31) of row r inside a 128-byte-swizzled tile
__device__ __forceinline__ uint32_t swz_e(int r, int e) { return swz(r, e >> 2) + (uint32_t)(e & 3) * 4u; }

__device__ __forceinline__ void tmem_st(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
      "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&r)[32]) { tmem_ld32(taddr, r); tmem_ld_wait_for(r); }
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&r)[16]) { tmem_ld16(taddr, r); tmem_ld_wait_for16(r); }

// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand is [M lanes][K columns] of fp32 words in tensor memory
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}

// The part of x that tf32 truncation drops, itself left unrounded: the tensor core truncates it again (error 2^-21 |x|, below
// the lo * lo term that a 3xTF32 product leaves out anyway).
__device__ __forceinline__ float lo_part(float x) { return x - tf32_hi(x); }

__device__ __forceinline__ float4 lo4(float4 v) { return make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w)); }

// Column sums over the rows of the tile are deferred: every tile adds a partially reduced copy of the thread's CW values
// into 8 registers (reduce-scatter butterfly over lane bits 16 [, 8]); finish8() completes the butterfly once, at the end
// of the kernel.  acc[i] of lane l belongs to column  (CW == 16 ? 8 * bit4(l) : 16 * bit4(l) + 8 * bit3(l)) + i.
template <int CW>
__device__ __forceinline__ void fold8(const float (&v)[CW], float (&acc)[8], int lane) {
  const bool up = (lane & 16) != 0;
  if (CW == 16) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const float send = up ? v[i] : v[i + 8];
      const float keep = up ? v[i + 8] : v[i];
      acc[i] += keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
  } else {
    float t[16];
#pragma unroll
    for (int i = 0; i < 16; i++) {
      const float send = up ? v[i] : v[i + 16];
      const float keep = up ? v[i + 16] : v[i];
      t[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
    const bool up8 = (lane & 8) != 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const float send = up8 ? t[i] : t[i + 8];
      const float keep = up8 ? t[i + 8] : t[i];
      acc[i] += keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
  }
}
// -> the warp's column sum; CW == 32: lane l holds column l, CW == 16: lanes 2c and 2c + 1 hold column c
template <int CW>
__device__ __forceinline__ float finish8(float (&acc)[8], int lane) {
  int off = (CW == 16) ? 8 : 4;
#pragma unroll
  for (int h = 4; h >= 1; h >>= 1, off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < h; i++) {
      const float send = up ? acc[i] : acc[i + h];
      const float keep = up ? acc[i + h] : acc[i];
      acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  if (CW == 16) acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 1);
  return acc[0];
}

// NQ column groups: thread = (operand row, group of CW = 64 / NQ columns); 128 * NQ threads
// DROP: training dropout (AFM.py:126,134).  The masks of a tile's two samples are drawn two tiles ahead, during the embedding
// scatter (where warps 10..15 have no items), one hash per lane of the last 8 warps, into Misc: the pair keep bits (one ballot
// per 32 pairs) and the column factors n_k.  With m_p (pairs) and n_k (columns): u_p is built
// with w~ = prediction_W n, the softmax uses od = sum a_p m_p u_p, c_r = g a_p m_p and ds = g a_p (m_p u_p - od), the direct
// term of dP is c_r w~ and the d prediction_W fold is scaled by n.  Everything downstream of ds is unchanged.
template <int NQ, bool DROP>
__global__ void __launch_bounds__(128 * NQ, 1) afm_fused_tc_kernel(const AfmArgs a, const int64_t n_tiles) {
  constexpr int CW = KD / NQ;
  constexpr int kThreads = 128 * NQ;
  // The three products are issued by lane 0 of three DIFFERENT warps, the last ones of the CTA: they have no share of the
  // embedding scatter (its items go to threads 0..351) while warp 0 has that plus the id bookkeeping, and every product
  // completes on its own mbarrier (a commit covers the issuing thread's MMAs), so nothing orders the issuers among themselves.
  // Issued by thread 0 the ~400 issue instructions of a tile were serial on the slowest warp: 3.62 -> 3.42 ms for one issuer
  // in the last warp.
  constexpr int kIssuer2 = kThreads - 32, kIssuer3 = kThreads - 64, kIssuer1 = (NQ == 4) ? kThreads - 96 : kThreads - 32;
  extern __shared__ uint8_t smem_raw[];
  __shared__ float scratch[32];
  // 1024-byte alignment by an offset from the __shared__ symbol (not an integer round trip of the pointer): the compiler keeps
  // the address space and emits LDS / STS instead of generic LD / ST for every access below
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  Misc& mi = *reinterpret_cast<Misc*>(smem + oMisc);
  float* EsBuf = reinterpret_cast<float*>(smem + oE);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int F = a.F, P = a.P;
  const int quarter = warp & 3, cg = warp >> 2, c0 = cg * CW;
  const int row = quarter * 32 + lane;          // operand row / TMEM lane of this thread
  const int ss = row >> 6, pp = row & 63;       // sample slot, pair index
  const bool prow = pp < P;

  // ---- one-time setup: W tiles, small vectors, pair tables, TMEM ----
  for (int i = tid; i < KD * (KD / 4); i += kThreads) {
    const int k = i / (KD / 4), c = i % (KD / 4);           // W row k, float4 chunk c of the A columns
    const float4 w = __ldg(reinterpret_cast<const float4*>(a.W) + i);
    // W tiles (rows = k, contiguous a): B operand of dP = dZ . W^T
    *reinterpret_cast<float4*>(smem + oWn + (c >> 3) * kWTile + swz(k, c & 7)) = w;
    *reinterpret_cast<float4*>(smem + oWn + (2 + (c >> 3)) * kWTile + swz(k, c & 7)) = lo4(w);
    // W^T tiles (rows = a, contiguous k): B operand of Z = P . W
    const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int an = 4 * c + q;
      const uint32_t off = swz(an, (k & 31) >> 2) + (uint32_t)(k & 3) * 4u;
      *reinterpret_cast<float*>(smem + oWt + (k >> 5) * kWTile + off) = wv[q];
      *reinterpret_cast<float*>(smem + oWt + (2 + (k >> 5)) * kWTile + off) = tf32_lo(wv[q]);
    }
  }
  if (tid < KD) {
    mi.batt[tid] = __ldg(a.batt + tid); mi.pvec[tid] = __ldg(a.pvec + tid); mi.wpred[tid] = __ldg(a.wpred + tid);
    mi.gbatt[tid] = 0.f; mi.gp[tid] = 0.f; mi.gwp[tid] = 0.f;
  }
  if (tid == 0) {
    int p = 0;
    for (int i = 0; i < F; i++)
      for (int j = i + 1; j < F; j++) {                      // AFM.py:105-112: pairs i < j in lexicographic order
        mi.pi[p] = (unsigned char)i; mi.pj[p] = (unsigned char)j;
        mi.pidx[i][j] = (unsigned char)p; mi.pidx[j][i] = (unsigned char)p;
        p++;
      }
    mbar_init(&mi.bar1, 1);
    mbar_init(&mi.bar2, 1);
    mbar_init(&mi.bar3, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&mi.tmem, kTmemCols);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = mi.tmem;
  const uint32_t t_lane = tmem + ((uint32_t)(quarter * 32) << 16);
  const uint32_t sP = smem_u32(smem + oP), sZ = smem_u32(smem + oZ), sWt = smem_u32(smem + oWt), sWn = smem_u32(smem + oWn);
  const float b0 = a.b0 ? __ldg(a.b0) : 0.f;
  const int rep = a.hot.slot ? (int)(blockIdx.x % a.hot.n_rep) : 0;
  const bool has_hot = a.hot.slot != nullptr;
  float loss_acc = 0.f, gb0_acc = 0.f;
  float dwacc[CW];                  // this thread's share of dW: TMEM lane `row` (k = row & 63, x or lo part), its CW columns
  float gb8[8], gp8[8], gw8[8];     // deferred column sums: d attention_b, d attention_p, d prediction_W (fold8)
#pragma unroll
  for (int i = 0; i < CW; i++) dwacc[i] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; i++) { gb8[i] = 0.f; gp8[i] = 0.f; gw8[i] = 0.f; }

  // 16 warps: thread i < 2 F 16 owns the same (sample slot, field, 16-byte chunk) item of the staging and of the embedding
  // scatter in every tile -- its decomposition (two integer divisions by the runtime F) and the tile rows of its F - 1 pairs
  // are worked out once; rows are packed four per register
  const bool it_on = NQ == 4 && tid < 2 * F * (KD / 4);
  const int it_s2 = it_on ? tid / (F * (KD / 4)) : 0, it_rem = it_on ? tid % (F * (KD / 4)) : 0;
  const int it_f = it_rem / (KD / 4), it_c = it_rem % (KD / 4);
  uint32_t it_rows[3] = {0u, 0u, 0u};
  if (it_on) {
#pragma unroll
    for (int j = 0; j < kMaxF; j++)
      if (j < F && j != it_f) it_rows[j >> 2] |= (uint32_t)(it_s2 * kSlot + mi.pidx[it_f][j]) << (8 * (j & 3));
  }
  // ---- staging pipeline (three buffers): ids three tiles ahead, embedding rows + bias values + hot slots two tiles ahead ----
  // id bookkeeping (load the ids of a tile three tiles ahead, store them, sum the bias values) by a warp that has neither
  // scatter items nor an issuer role when there is one (16 warps: warp 12)
  constexpr int kBook0 = (NQ == 4) ? kThreads - 128 : 0;
  const int bt = tid - kBook0;                  // 0 .. 2F-1: (sample slot, field) of this thread's id
  auto load_id = [&](int64_t t) {
    if (bt < 0 || bt >= 2 * F || t >= n_tiles) return -1;
    const int64_t s = 2 * t + bt / F;
    return (s < a.B) ? __ldg(a.idx + s * F + bt % F) : -1;
  };
  auto stage_rows = [&](int buf, int islot) {   // rows of the tile whose ids are in mi.ids[islot] -> EsBuf[buf], biasv[buf], hslot[buf]
    float* Es = EsBuf + buf * (kEBytes / 4);
    for (int i = tid; i < 2 * F * (KD / 4); i += kThreads) {
      int s2, f, c;
      if (NQ == 4) { s2 = it_s2; f = it_f; c = it_c; }
      else { s2 = i / (F * (KD / 4)); const int rem = i % (F * (KD / 4)); f = rem / (KD / 4); c = rem % (KD / 4); }
      const int id = mi.ids[islot][s2][f];
      float* dst = Es + (s2 * kMaxF + f) * kEP + 4 * c;
      if (id >= 0) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(a.V + (size_t)id * KD + 4 * c) : "memory");
        if (c == 0 && a.bias) ldgsts4(&mi.biasv[buf][s2][f], a.bias + id);
        if (c == 1 && has_hot) ldgsts4(&mi.hslot[buf][s2][f], a.hot.slot + id);
      } else {
        *reinterpret_cast<float4*>(dst) = f4_zero();
        if (c == 0) mi.biasv[buf][s2][f] = 0.f;
      }
    }
    ldgsts_commit();
  };
  // this thread's CW pair products of the tile staged in Es (zero for the padding rows of a slot)
  const int off_i = (ss * kMaxF + mi.pi[prow ? pp : 0]) * kEP + c0, off_j = (ss * kMaxF + mi.pj[prow ? pp : 0]) * kEP + c0;
  auto pair_products = [&](const float* Es, float (&pr)[CW], float scale) {
    const float* ei = Es + off_i;
    const float* ej = Es + off_j;
    const float m = prow ? scale : 0.f;
#pragma unroll
    for (int i = 0; i < CW; i += 4) {
      const float4 x = *reinterpret_cast<const float4*>(ei + i), y = *reinterpret_cast<const float4*>(ej + i);
      pr[i] = m * (x.x * y.x); pr[i + 1] = m * (x.y * y.y); pr[i + 2] = m * (x.z * y.z); pr[i + 3] = m * (x.w * y.w);
    }
  };
  // DROP: the masks of the tile `tile` (two samples) -> abits / nvec [pr]; warp-uniform, called by every thread
  auto stage_masks = [&](int64_t tile, int pr) {
    constexpr int w0 = kThreads / 32 - 8;
    if constexpr (DROP) if (warp >= w0) {
      const int w8 = warp - w0, sl = (w8 >> 1) & 1, wd = w8 & 1;
      const int64_t smp2 = 2 * tile + sl;
      if (w8 < 4) {
        mi.nvec[pr][sl][32 * wd + lane] = afm_mask_vec(a, splitmix64(a.drop_seed), smp2, 32 * wd + lane) / a.keep_vec;
      } else {
        const uint32_t bits = __ballot_sync(0xffffffffu, afm_mask_att(a, smp2, 32 * wd + lane) != 0.f);
        if (lane == 0) mi.abits[pr][sl][wd] = bits;
      }
    }
  };
  // w~_i = prediction_W n_i of this thread's column i in the tile of parity pr
  auto wtilde = [&](int pr, int i) {
    if constexpr (DROP) return mi.wpred[c0 + i] * mi.nvec[pr][ss][c0 + i];
    else return mi.wpred[c0 + i];
  };
  // P rows of a tile -> TMEM (x and lo): the A operand of GEMM 1
  auto build_p_tmem = [&](const float* Es, int par) {
    float pr[CW];
    uint32_t rx[CW], rl[CW];
    pair_products(Es, pr, 1.f);
    float up = 0.f;
#pragma unroll
    for (int i = 0; i < CW; i++) {
      rx[i] = __float_as_uint(pr[i]); rl[i] = __float_as_uint(lo_part(pr[i]));
      up = fmaf(wtilde(par, i), pr[i], up);                              // u_p = prediction_W . P_p (AFM.py:138-139, per pair)
    }
    mi.u_part[par][cg][row] = up;
    tmem_st(t_lane + cPX + c0, rx);
    tmem_st(t_lane + cPL + c0, rl);
    tmem_st_wait();
  };
  auto issue_gemm1 = [&]() {                // Z = P . W (3xTF32): A = P from TMEM, B = W^T tiles
    const uint32_t idesc = make_idesc_tf32(kRows, KD);
#pragma unroll
    for (int kb = 0; kb < 2; kb++)
#pragma unroll
      for (int k4 = 0; k4 < 4; k4++) {
        const uint32_t o = k4 * 32, kc = kb * 32 + k4 * 8;          // byte offset inside the B tile row / A column offset
        const uint32_t bx = sWt + kb * kWTile + o, bl = sWt + (2 + kb) * kWTile + o;
        umma_tf32_ts(tmem + cZ, tmem + cPL + kc, make_sdesc(bx), idesc, (kb | k4) ? 1u : 0u);
        umma_tf32_ts(tmem + cZ, tmem + cPX + kc, make_sdesc(bl), idesc, 1u);
        umma_tf32_ts(tmem + cZ, tmem + cPX + kc, make_sdesc(bx), idesc, 1u);
      }
    umma_commit(&mi.bar1);
  };
  const int64_t g_tiles = gridDim.x;
  int buf = 0, par = 0, islot = 0;      // staging buffer (mod 3), u_part parity, ids ring slot (mod 4) of the current tile
  {
    const int id0 = load_id(blockIdx.x), id1 = load_id((int64_t)blockIdx.x + g_tiles);
    if (bt >= 0 && bt < 2 * F) { mi.ids[0][bt / F][bt % F] = id0; mi.ids[1][bt / F][bt % F] = id1; }
    if constexpr (DROP) {
      stage_masks(blockIdx.x, 0);
      stage_masks((int64_t)blockIdx.x + g_tiles, 1);
    }
    if (tid < 2 * (kMaxF + 1)) {
      const int s2 = tid / (kMaxF + 1), f = tid % (kMaxF + 1);
#pragma unroll
      for (int q = 0; q < 3; q++) { mi.biasv[q][s2][f] = 0.f; mi.hslot[q][s2][f] = -1; }
    }
    __syncthreads();
    stage_rows(0, 0);
    stage_rows(1, 1);
    ldgsts_wait<1>();                       // the first tile's rows
    __syncthreads();
    build_p_tmem(EsBuf, 0);
    tc_fence_before();
    __syncthreads();
    if (tid == kIssuer1) { tc_fence_after(); issue_gemm1(); }
  }
  int id_reg = load_id((int64_t)blockIdx.x + 2 * g_tiles);      // ids of the tile after next, stored at the top of the next tile
  uint32_t ph1 = 0, ph2 = 0;

  // Software pipeline: GEMM 1 of tile t+1 is issued before the embedding scatter of tile t and completes behind it; its
  // operand (the P rows of tile t+1 in TMEM) is built behind GEMM 2 / 3 of tile t.
  for (int64_t t = blockIdx.x; t < n_tiles; t += g_tiles) {
    const int nb = (buf == 2) ? 0 : buf + 1, nnb = (nb == 2) ? 0 : nb + 1;
    const float* Es = EsBuf + buf * (kEBytes / 4);
    const bool has_next = t + g_tiles < n_tiles;
    // No barrier here: warps that are done with the previous tile's scatter start on this tile's PT tiles while the others
    // finish.  Everything the scatter still reads (its staged rows, hot slots, ids, the dP rows, mi.g) is next written after
    // barrier (3) below, except the ids -- hence the four-deep ring: slot + 2 was last read two tiles ago.
    if (bt >= 0 && bt < 2 * F) mi.ids[(islot + 2) & 3][bt / F][bt % F] = id_reg;
    id_reg = load_id(t + 3 * g_tiles);
    const int64_t smp = 2 * t + ss;
    const float label = (smp < a.B) ? __ldg(a.labels + smp) : 0.f;
    if (bt == 30 || bt == 31) {                  // two more lanes of the bookkeeping warp (2 F <= 22)
      float bs = 0.f;
      for (int f = 0; f < F; f++) bs += mi.biasv[buf][bt - 30][f];
      mi.bsum[bt - 30] = bs;
    }
    // ---- phase 1: the K-major PT tiles (A of GEMM 3; GEMM 3 of the previous tile is complete) ----
    {
      float pr[CW];
      pair_products(Es, pr, 1.f);
      uint8_t* pt = smem + oP + (uint32_t)quarter * kTile;             // r block = quarter, column of the tile row = lane
#pragma unroll
      for (int i = 0; i < CW; i++) {
        const int k = c0 + i;
        *reinterpret_cast<float*>(pt + swz_e(k, lane)) = pr[i];
        *reinterpret_cast<float*>(pt + swz_e(KD + k, lane)) = lo_part(pr[i]);
      }
    }
    mbar_wait(&mi.bar1, ph1, nullptr);      // GEMM 1 of this tile (issued one tile ago)
    ph1 ^= 1;
    tc_fence_after();

    // ---- epilogue 1: logits ----
    {
      uint32_t r[CW];
      tmem_ld(t_lane + cZ + c0, r);
      float sp = 0.f;
#pragma unroll
      for (int i = 0; i < CW; i++) {
        const float zi = __uint_as_float(r[i]) + mi.batt[c0 + i];                // AFM.py:117-123
        sp = fmaf(fmaxf(zi, 0.f), mi.pvec[c0 + i], sp);
      }
      mi.s_part[cg][row] = sp;
    }
    ldgsts_wait<0>();           // the next tile's rows (staged one tile ago)
    __syncthreads();
    if (t + 2 * g_tiles < n_tiles) stage_rows(nnb, (islot + 2) & 3);
    // Every warp works out the softmax of its sample slot by itself: lane l looks at the slot's pairs l and l + 32.
    float c_r, ds;
    {
      const int rlo = ss * kSlot + lane, rhi = rlo + 32;
      float s_lo = mi.s_part[0][rlo], s_hi = mi.s_part[0][rhi], u_lo = mi.u_part[par][0][rlo], u_hi = mi.u_part[par][0][rhi];
#pragma unroll
      for (int q = 1; q < NQ; q++) {
        s_lo += mi.s_part[q][rlo]; s_hi += mi.s_part[q][rhi];
        u_lo += mi.u_part[par][q][rlo]; u_hi += mi.u_part[par][q][rhi];
      }
      const bool v_lo = lane < P, v_hi = lane + 32 < P;
      float mx = fmaxf(v_lo ? s_lo : -INFINITY, v_hi ? s_hi : -INFINITY);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      const float e_lo = v_lo ? expf(s_lo - mx) : 0.f, e_hi = v_hi ? expf(s_hi - mx) : 0.f;   // AFM.py:125 softmax over the pairs
      float m_lo = 1.f, m_hi = 1.f;                           // m_p of the pairs lane and lane + 32 (DROP)
      if constexpr (DROP) {
        const float m_on = 1.f / a.keep_att;
        m_lo = ((mi.abits[par][ss][0] >> lane) & 1u) ? m_on : 0.f;
        m_hi = ((mi.abits[par][ss][1] >> lane) & 1u) ? m_on : 0.f;
        u_lo *= m_lo; u_hi *= m_hi;                           // m_p u_p
      }
      float d0 = e_lo, d1 = e_hi, n0 = e_lo * u_lo, n1 = e_hi * u_hi;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        d0 += __shfl_xor_sync(0xffffffffu, d0, o); d1 += __shfl_xor_sync(0xffffffffu, d1, o);
        n0 += __shfl_xor_sync(0xffffffffu, n0, o); n1 += __shfl_xor_sync(0xffffffffu, n1, o);
      }
      const float den = d0 + d1;
      const float od = (n0 + n1) / den;                       // sum_p a_p (prediction_W . P_p) = prediction_W . afm, AFM.py:130-139
      const float att = ((pp < 32) ? e_lo : e_hi) / den;
      const float u_r = (pp < 32) ? u_lo : u_hi;            // DROP: m_p u_p
      float g = 0.f;
      if (smp < a.B) {
        const float out = (od + mi.bsum[ss]) + b0;            // AFM.py:142
        const float diff = label - out;
        g = -diff;
        if (pp == 0 && cg == 0) {
          loss_acc += 0.5f * diff * diff;                     // AFM.py:146 tf.nn.l2_loss
          gb0_acc += g;
          if (a.out) a.out[smp] = out;
        }
      }
      if (pp == 0 && cg == 0) mi.g[ss] = g;
      if constexpr (DROP) {                                   // d a_p = g m_p u_p; ds = a (da - sum a da)
        c_r = (g * att) * ((pp < 32) ? m_lo : m_hi);
        ds = (g * att) * (u_r - od);
      } else {
        c_r = g * att;                                        // d afm . P_p = g * u_p; softmax backward: ds = a (da - sum a da)
        ds = c_r * (u_r - od);
      }
    }
    // dZ = ds * p * relu'(Z + b) -> TMEM (A of GEMM 2) and the K-major dZT tiles (B of GEMM 3)
    float dz[CW], hp[CW];
    {
      uint32_t rx[CW], rl[CW];
      uint8_t* zt = smem + oZ + (uint32_t)quarter * kWTile;             // dZT x tiles: r block = quarter, column = lane
      tmem_ld(t_lane + cZ + c0, rx);                                    // the logits again (cheaper than CW live registers)
#pragma unroll
      for (int i = 0; i < CW; i++) {
        const float zi = __uint_as_float(rx[i]) + mi.batt[c0 + i];
        const bool on = zi > 0.f;
        dz[i] = on ? ds * mi.pvec[c0 + i] : 0.f;
        hp[i] = on ? ds * zi : 0.f;                                     // d p += ds * relu(Z + b)
        const float lo = lo_part(dz[i]);
        rx[i] = __float_as_uint(dz[i]); rl[i] = __float_as_uint(lo);
        const int an = c0 + i;
        *reinterpret_cast<float*>(zt + swz_e(an, lane)) = dz[i];
        *reinterpret_cast<float*>(zt + 4 * kWTile + swz_e(an, lane)) = lo;
      }
      tmem_st(t_lane + cZX + c0, rx);
      tmem_st(t_lane + cZL + c0, rl);
      tmem_st_wait();
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (tid == kIssuer2) {
      tc_fence_after();
      const uint32_t idesc = make_idesc_tf32(kRows, KD);
#pragma unroll
      for (int ab = 0; ab < 2; ab++)
#pragma unroll
        for (int k4 = 0; k4 < 4; k4++) {
          const uint32_t o = k4 * 32, kc = ab * 32 + k4 * 8;
          const uint32_t bx = sWn + ab * kWTile + o, bl = sWn + (2 + ab) * kWTile + o;
          umma_tf32_ts(tmem + cDP, tmem + cZL + kc, make_sdesc(bx), idesc, (ab | k4) ? 1u : 0u);
          umma_tf32_ts(tmem + cDP, tmem + cZX + kc, make_sdesc(bl), idesc, 1u);
          umma_tf32_ts(tmem + cDP, tmem + cZX + kc, make_sdesc(bx), idesc, 1u);
        }
      umma_commit(&mi.bar2);
    }
    if (tid == kIssuer3) {
      tc_fence_after();
      const uint32_t idesc = make_idesc_tf32(kRows, KD);
      // dW: reduction over the 128 tile rows = 4 r blocks x 4 k-steps of 8; A = [PT x ; PT lo] (M = 128), B = dZT x, dZT lo
#pragma unroll
      for (int rb = 0; rb < 4; rb++)
#pragma unroll
        for (int k4 = 0; k4 < 4; k4++) {
          const uint32_t o = k4 * 32;
          const uint64_t ad = make_sdesc(sP + rb * kTile + o);
          umma_tf32(tmem + cDW, ad, make_sdesc(sZ + rb * kWTile + o), idesc, (rb | k4) ? 1u : 0u);
          umma_tf32(tmem + cDW, ad, make_sdesc(sZ + (4 + rb) * kWTile + o), idesc, 1u);
        }
      umma_commit(&mi.bar3);
    }
    // behind GEMM 2 / 3: the column sums over the tile rows (d b = sum dZ, d p, d prediction_W = sum g a_p P_p), deferred,
    // and the P rows of the next tile -> TMEM
    fold8<CW>(dz, gb8, lane);
    fold8<CW>(hp, gp8, lane);
    pair_products(Es, dz, c_r);
    if constexpr (DROP) {
#pragma unroll
      for (int i = 0; i < CW; i++) dz[i] *= mi.nvec[par][ss][c0 + i];
    }
    fold8<CW>(dz, gw8, lane);
    if (has_next) build_p_tmem(EsBuf + nb * (kEBytes / 4), par ^ 1);
    mbar_wait(&mi.bar2, ph2, nullptr);      // GEMM 2
    tc_fence_after();

    // ---- epilogue 2: dP rows (+ the direct path a_p * d afm = g a_p prediction_W) -> shared memory, once GEMM 3 is done with
    //      the dZT tiles ----
    {
      uint32_t r[CW];
      tmem_ld(t_lane + cDP + c0, r);
#pragma unroll
      for (int i = 0; i < CW; i++) r[i] = __float_as_uint(fmaf(c_r, wtilde(par, i), __uint_as_float(r[i])));
      mbar_wait(&mi.bar3, ph2, nullptr);    // GEMM 3
      ph2 ^= 1;
      tc_fence_after();
      float* dst = reinterpret_cast<float*>(smem + oZ) + row * KD;
#pragma unroll
      for (int c = 0; c < CW / 4; c++)
        *reinterpret_cast<float4*>(dst + 4 * ((cg * (CW / 4) + c) ^ (row & 15))) =
            make_float4(__uint_as_float(r[4 * c]), __uint_as_float(r[4 * c + 1]), __uint_as_float(r[4 * c + 2]), __uint_as_float(r[4 * c + 3]));
      tmem_ld(t_lane + cDW + c0, r);                          // this tile's dW partial sum -> registers (two-level accumulation)
#pragma unroll
      for (int i = 0; i < CW; i++) dwacc[i] += __uint_as_float(r[i]);
    }
    tc_fence_before();
    __syncthreads();
    if (tid == kIssuer1 && has_next) { tc_fence_after(); issue_gemm1(); }      // GEMM 1 of the next tile runs behind the scatter below
    // the masks of tile t + 2 into parity par: its last reader (this tile's epilogue 2) is behind the barrier above, its first
    // reader (the P rows of tile t + 2, built in the next tile) behind the next tile's barrier (1)
    if constexpr (DROP) stage_masks(t + 2 * g_tiles, par);
    // dE_f = sum_{j != f} dP_(f,j) * E_j ; one vector reduction per 16 bytes of the gradient row
    for (int i = tid; i < 2 * F * (KD / 4); i += kThreads) {
      int s2, f, c;
      if (NQ == 4) { s2 = it_s2; f = it_f; c = it_c; }
      else { s2 = i / (F * (KD / 4)); const int rem = i % (F * (KD / 4)); f = rem / (KD / 4); c = rem % (KD / 4); }
      const int id = mi.ids[islot][s2][f];
      if (id < 0) continue;
      float4 acc = f4_zero();
#pragma unroll
      for (int j = 0; j < kMaxF; j++) {                       // unrolled: the loads of all terms are in flight together
        if (j >= F || j == f) continue;
        const int r2 = (NQ == 4) ? (int)((it_rows[j >> 2] >> (8 * (j & 3))) & 0xFFu) : s2 * kSlot + mi.pidx[f][j];
        const float4 dp = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(smem + oZ) + r2 * KD + 4 * (c ^ (r2 & 15)));
        const float4 e = *reinterpret_cast<const float4*>(Es + (s2 * kMaxF + j) * kEP + 4 * c);
        acc.x = fmaf(dp.x, e.x, acc.x); acc.y = fmaf(dp.y, e.y, acc.y); acc.z = fmaf(dp.z, e.z, acc.z); acc.w = fmaf(dp.w, e.w, acc.w);
      }
      float* dst = a.gV + (size_t)id * KD;
      const int hs = has_hot ? mi.hslot[buf][s2][f] : -1;
      if (hs >= 0) dst = a.hot.ghot + ((size_t)rep * a.hot.n_hot + hs) * KD;
      red_add_v4(dst + 4 * c, acc);
      if (c == 0) {
        if (a.gbias) {
          float* pb = (hs >= 0 && a.hot.ghot_bias != nullptr) ? a.hot.ghot_bias + (size_t)rep * a.hot.n_hot + hs : a.gbias + id;
          atomicAdd(pb, mi.g[s2]);
        }
        if (a.touch_stamp) a.touch_stamp[id] = a.stamp;      // compacted into the touched-row list afterwards
      }
    }
    buf = nb;
    par ^= 1;
    islot = (islot + 1) & 3;
  }

  ldgsts_wait<0>();
  tc_fence_before();
  __syncthreads();
  // ---- flush the accumulators: dW[k][a] = D[k][a] + D[64 + k][a] (x and lo rows land on the same element) ----
  {
    float* dst = a.gW + (size_t)(row & 63) * KD + c0;
#pragma unroll
    for (int i = 0; i < CW; i++)
      if (dwacc[i] != 0.f) atomicAdd(dst + i, dwacc[i]);
  }
  {
    const float cb = finish8<CW>(gb8, lane), cp = finish8<CW>(gp8, lane), cw = finish8<CW>(gw8, lane);
    const int col = c0 + ((CW == 16) ? (lane >> 1) : lane);
    if (CW == 32 || (lane & 1) == 0) {
      atomicAdd(&mi.gbatt[col], cb); atomicAdd(&mi.gp[col], cp); atomicAdd(&mi.gwp[col], cw);
    }
  }
  __syncthreads();
  if (tid < KD) {
    atomicAdd(a.gbatt + tid, mi.gbatt[tid]);
    atomicAdd(a.gp + tid, mi.gp[tid]);
    atomicAdd(a.gwpred + tid, mi.gwp[tid]);
  }
  {
    const float bl = block_sum(loss_acc, scratch);
    write_partial(a.loss_partials, bl);
    const float bg = block_sum(gb0_acc, scratch);
    if (tid == 0 && a.gb0 != nullptr && bg != 0.f) atomicAdd(a.gb0, bg);
  }
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, kTmemCols);
}

}  // namespace aft

template <bool DROP>
static bool configure_fused_tc() {
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(aft::afm_fused_tc_kernel<4, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)aft::kSmemBytes) != cudaSuccess ||
        cudaFuncSetAttribute(aft::afm_fused_tc_kernel<2, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)aft::kSmemBytes) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    configured = true;
  }
  return true;
}

int dispatch_afm_fused_tc(const AfmArgs& a, int64_t M, cudaStream_t st, bool drop) {
  if (a.K != aft::KD || a.A != aft::KD || a.F > aft::kMaxF || a.F < 2 || a.P > aft::kSlot) return 1;
  const char* env = getenv("HHFM_AFM_TC");               // 0 = fp32 CUDA-core kernels (A/B runs, tests of both paths)
  if (env && env[0] == '0') return 1;
  if (!(drop ? configure_fused_tc<true>() : configure_fused_tc<false>())) return 1;
  const int groups = (env && env[0] == '2') ? 2 : 4;      // column groups per row: 4 = 16 warps (default), HHFM_AFM_TC=2: 8 warps
  const int64_t n_tiles = (a.B + 1) / 2;
  int grid = sm_count();
  if (grid > kPartials) grid = kPartials;
  if ((int64_t)grid > n_tiles) grid = (int)n_tiles;
  if (drop) {
    if (groups == 4) aft::afm_fused_tc_kernel<4, true><<<grid, 512, aft::kSmemBytes, st>>>(a, n_tiles);
    else aft::afm_fused_tc_kernel<2, true><<<grid, 256, aft::kSmemBytes, st>>>(a, n_tiles);
  } else {
    if (groups == 4) aft::afm_fused_tc_kernel<4, false><<<grid, 512, aft::kSmemBytes, st>>>(a, n_tiles);
    else aft::afm_fused_tc_kernel<2, false><<<grid, 256, aft::kSmemBytes, st>>>(a, n_tiles);
  }
  int rc = check_launch("afm_fused_tc_kernel");
  if (rc != HHFM_OK) return rc;
  if (a.touch_stamp != nullptr) rc = launch_touched_compact(a.touch_stamp, a.stamp, M, a.touched_rows, a.touched_count, st);
  return rc;
}

}  // namespace hhfm
