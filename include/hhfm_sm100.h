/*
 * hhfm_sm100.h -- C ABI of libhhfm_sm100.so: the B200 (sm_100a) replacement for the factorization-machine
 * hot path of data-man-34/HHFM (Newcode/*.py).
 *
 * The reference has no native layer: its "kernels" are the TensorFlow-1.x ops instantiated by the graphs in
 * Newcode/{FM,MF,AFM,DFM,OurModel7,BPR}.py and executed by `sess.run` (FM.py:168-171).  Each entry point
 * below names the reference graph lines (file:line under /root/reference) whose TF ops it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  All device pointers are CALLER-OWNED (torch tensors on the
 *     host side); the library never allocates or frees device memory.  Scratch is passed in; sizes come from
 *     the hhfm_*_len / hhfm_workspace_bytes_* queries.
 *   - Every device entry point takes a CUDA stream and is stream-ordered / asynchronous, re-entrant across
 *     streams, and keeps no global mutable state (the last-error string is thread-local).
 *   - Return value: HHFM_OK (0) or a negative hhfm_status.  `hhfm_last_error()` describes the last failure
 *     on the calling thread.  No exception crosses the ABI.  There is NO CPU fallback: without a CUDA device
 *     the device entry points return HHFM_ERR_LAUNCH.
 *   - dtype: float32 values, int32 ids (FM.py:89), shapes as int64_t.  Embedding tables are row-major
 *     [M, K] with K % 4 == 0, K <= 512, 16-byte aligned.
 *   - Gradient buffers are accumulated into (+=) with red.global.add.v4.f32; the caller (or the optimizer
 *     entry points with zero_grad=1) keeps them zero between steps.
 */
#ifndef HHFM_SM100_H
#define HHFM_SM100_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* hhfm_stream_t; /* cudaStream_t */

typedef enum {
  HHFM_OK = 0,
  HHFM_ERR_BAD_ARG = -1,
  HHFM_ERR_UNSUPPORTED = -2,
  HHFM_ERR_LAUNCH = -3
} hhfm_status;

/* Pooling1C / Pooling1T / Pooling1F of OurModel7.py:14-19 (tf.reduce_sum | reduce_max | reduce_mean) */
typedef enum { HHFM_POOL_SUM = 0, HHFM_POOL_MAX = 1, HHFM_POOL_MEAN = 2 } hhfm_pool;

/* optimizer kinds: FM.py:129-136 (tf.train.{Adagrad,Adam,Momentum,GradientDescent}Optimizer) */
typedef enum { HHFM_OPT_ADAGRAD = 0, HHFM_OPT_ADAM = 1, HHFM_OPT_MOMENTUM = 2, HHFM_OPT_SGD = 3 } hhfm_opt;

/* DeepFM options (K8 *_mode entry points), OR-ed: use_fm=False, use_deep=False, loss_type='logloss'.  0 = the reference's
 * default (both parts, mse).  NO_FM | NO_DEEP and unknown bits are rejected. */
typedef enum { HHFM_DFM_NO_FM = 1, HHFM_DFM_NO_DEEP = 2, HHFM_DFM_LOGLOSS = 4 } hhfm_dfm_mode;

/* top-N query kinds */
typedef enum {
  HHFM_QUERY_USER = 0, /* q = V[user]                      BPR.py:132, MF.py:145          */
  HHFM_QUERY_FM = 1,   /* q = V[user]+Fc, Fc = sum ctx     FM.py:174-177                  */
  HHFM_QUERY_HHFM = 2  /* q = hybrid feature               OurModel7.py:232-292           */
} hhfm_query;

int hhfm_abi_version(void);
const char* hhfm_last_error(void);
/* number of float slots every `loss_partials` / `sq_partials` argument must provide */
int64_t hhfm_partials_len(void);

/* ------------------------------------------------------------------------------------------------
 * K0  host-side batch packing (CPU threads; dst may be pinned host memory).
 * Replaces the numpy slicing that feeds `feed_dict` (FM.py:251-256, OurModel7.py:373-385): int64 (or int32)
 * id columns are narrowed to int32 and written into a row-major record buffer with a caller-chosen row
 * stride, so one sample's ids are contiguous and 16-byte aligned for the device kernels.
 * Ids outside [0, id_limit) make the call fail with HHFM_ERR_BAD_ARG (TF's gather would raise).
 * ------------------------------------------------------------------------------------------------ */
int hhfm_pack_ids_i64(const int64_t* src, int64_t rows, int64_t cols, int64_t src_row_stride,
                      int32_t* dst, int64_t dst_row_stride, int64_t dst_col0, int64_t id_limit, int nthreads);
int hhfm_pack_ids_i32(const int32_t* src, int64_t rows, int64_t cols, int64_t src_row_stride,
                      int32_t* dst, int64_t dst_row_stride, int64_t dst_col0, int64_t id_limit, int nthreads);
/* fill columns [dst_col0, dst_col0+cols) of every record with `value` (padding = -1) */
int hhfm_pack_fill_i32(int32_t* dst, int64_t rows, int64_t cols, int64_t dst_row_stride, int64_t dst_col0,
                       int32_t value, int nthreads);
/* general CSR: ids [rows, cols] (+ optional values) -> row_ptr int32[rows+1], col int32[rows*cols],
 * val f32[rows*cols] (val/src_val may both be NULL => implicit 1.0, the reference's one-hot fields). */
int hhfm_pack_csr_i64(const int64_t* src, const float* src_val, int64_t rows, int64_t cols, int64_t src_row_stride,
                      int32_t* row_ptr, int32_t* col, float* val, int64_t id_limit, int nthreads);

/* Fused, pipelined packer + upload (the path Model.partial_fit uses): the id blocks `parts` (column groups of one batch,
 * int64 or int32, e.g. X | F1 | Y of OurModel7.py:374-385) are narrowed and interleaved into [rows, stride] records
 * (padding = -1) by a persistent host thread pool, chunk by chunk, and every finished chunk is sent with
 * cudaMemcpyAsync on `stream` while the next one is being packed.  When id_limit <= 65535 the wire format is uint16
 * (half the PCIe bytes) and a device kernel widens it into the int32 records the kernels read.
 *   host_staging: pinned host memory, hhfm_pack_upload_staging_bytes() bytes; dev_staging: device scratch of the same
 *   size (only used by the 16-bit format, may be NULL otherwise); dev_records: int32 [rows, stride] on the device.
 * Stream-ordered: returns after the last copy is enqueued; host_staging may be reused after the stream passes it. */
typedef struct hhfm_pack_part {
  const void* data;      /* [rows, cols] ids, row-major */
  int64_t cols;
  int64_t row_stride;    /* elements between consecutive rows */
  int32_t elem_bytes;    /* 8 = int64, 4 = int32 */
  int32_t reserved;
} hhfm_pack_part;
int64_t hhfm_pack_upload_staging_bytes(int64_t rows, int64_t stride, int64_t id_limit);
int hhfm_pack_upload_records(const hhfm_pack_part* parts, int32_t n_parts, int64_t rows, int64_t stride, int64_t id_limit,
                             void* host_staging, void* dev_staging, int32_t* dev_records, int32_t nthreads,
                             hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K1  FM / MF: gather + second-order interaction (+ squared loss + backward scatter)
 *   out[s] = sum_k 0.5((sum_f e_f)^2 - sum_f e_f^2) + sum_f val_f*bias[x_f] + b0,  e_f = val_f * V[x_f]
 *   FM.py:99-120 (embedding_lookup, reduce_sum, square, subtract, add_n); DFM.py:104-122 second order.
 *   interaction = 1 selects MF.py:81-92: out = sum_k V[x_0]*V[x_1] (first two ids, no bias).
 * Batch layout: CSR.  row_ptr == NULL means fixed width F (row s owns col[s*F .. s*F+F)); val == NULL
 * means all values 1.0.  bias / b0 may be NULL (treated as 0).  b0 is a device scalar.
 * ------------------------------------------------------------------------------------------------ */
int hhfm_fm_fwd(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B, int64_t F,
                const float* V, const float* bias, const float* b0, int64_t M, int64_t K, int32_t interaction,
                float* out, hhfm_stream_t stream);

/* Fused training pass: forward, loss = 0.5*sum(y-out)^2 (FM.py:123-126), and TF-autodiff-equivalent
 * backward: gV[x_f] += g*val_f*(S - e_f), gbias[x_f] += g*val_f, gb0 += g, g = out - y.
 * Duplicate ids (inside a row or across rows) are summed like UnsortedSegmentSum.
 *   out            [B] nullable
 *   gV             [M,K], accumulated into
 *   gbias          [M] nullable;  gb0 [1] nullable
 *   loss_partials  [hhfm_partials_len()]: per-CTA partial sums, reduce with hhfm_loss_finalize
 *   touch_stamp    [M] nullable: if given, every row whose stamp != `stamp` is stamped and appended to
 *                  touched_rows (capacity M) with touched_count[0] incremented -> feeds the *_rows optimizers
 *   hot_slot       [M] nullable: two-level scatter for rows that many samples share (low-cardinality columns,
 *                  Zipf heads).  hot_slot[row] = s >= 0 sends that row's reductions to replica (group % n_rep) of
 *                  ghot [n_rep, n_hot, K] (ghot_bias [n_rep, n_hot]) instead of gV / gbias, so they do not
 *                  serialise on one L2 slice; call hhfm_hot_fold before the optimizer.  -1 = cold row.
 *   deterministic  1 = one warp, program-order accumulation (bit-reproducible; test mode)              */
int hhfm_fm_fwd_bwd_sqloss(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B, int64_t F,
                           const float* V, const float* bias, const float* b0, int64_t M, int64_t K,
                           int32_t interaction, const float* labels, float* out, float* gV, float* gbias, float* gb0,
                           float* loss_partials, int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows,
                           int32_t* touched_count, const int32_t* hot_slot, float* ghot, float* ghot_bias,
                           int32_t n_rep, int32_t n_hot, int32_t deterministic, hhfm_stream_t stream);
/* The same step with tf.nn.dropout on the [B, K] interaction vector before the sum over k (FM.py:114, MF.py:87; the
 * reference's MF default is keep = 0.7): element (s, k) is kept iff u24(splitmix64(seed ^ splitmix64(s*0x100000001B3 + k)))
 * * 2^-24 < keep, kept elements are divided by keep.  keep = 1 is the call above.  Counter-based masks: statistically
 * TF's dropout, not its random stream; restated bit-exactly by the oracle (dropout_mask_hashed). */
int hhfm_fm_fwd_bwd_sqloss_dropout(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B, int64_t F,
                           const float* V, const float* bias, const float* b0, int64_t M, int64_t K,
                           int32_t interaction, const float* labels, float* out, float* gV, float* gbias, float* gb0,
                           float* loss_partials, int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows,
                           int32_t* touched_count, const int32_t* hot_slot, float* ghot, float* ghot_bias,
                           int32_t n_rep, int32_t n_hot, int32_t deterministic, float keep, uint64_t drop_seed, hhfm_stream_t stream);

/* FM training step with batch normalisation of the interaction vector (FM.py:111-112, batch_norm=1; tf.contrib.layers
 * .batch_norm with center, scale, is_training=True), before the dropout of the call above:
 *   x = 0.5 (S^2 - sum_f e_f^2), y = gamma (x - mu) / sqrt(var + eps) + beta, out = sum_k y / keep * m + sum_f b[x_f] + b0,
 * mu and var (biased) over the batch per column.  In the same step moving_mean -= (1 - decay) (moving_mean - mu) and
 * moving_var -= (1 - decay) (moving_var - var * B / max(B - 1, 1)).  dgamma / dbeta [K] are WRITTEN (not accumulated);
 * gV, gbias, gb0, the loss partials, the hot replicas and the touched-row list as in hhfm_fm_fwd_bwd_sqloss.
 * Fixed-width rows only (row_ptr = val = NULL) and interaction = 0; gamma, beta, moving_mean, moving_var 16-byte aligned.
 * eps > 0 (the reference: 1e-3), decay in [0, 1) (0.9).  workspace: hhfm_workspace_bytes_fm_bn(B, K) bytes, caller-owned,
 * 16-byte aligned.  Batch statistics, loss, dgamma, dbeta, gb0 and the moving statistics are fixed-order reductions
 * (bit-identical from run to run); deterministic = 1 also makes the row scatter one warp in program order. */
int hhfm_fm_bn_fwd_bwd_sqloss(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B, int64_t F,
                              const float* V, const float* bias, const float* b0, int64_t M, int64_t K,
                              int32_t interaction, const float* labels, float* out, float* gV, float* gbias, float* gb0,
                              float* loss_partials, int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows,
                              int32_t* touched_count, const int32_t* hot_slot, float* ghot, float* ghot_bias,
                              int32_t n_rep, int32_t n_hot, int32_t deterministic, float keep, uint64_t drop_seed,
                              const float* gamma, const float* beta, float* moving_mean, float* moving_var, float* dgamma,
                              float* dbeta, float eps, float decay, void* workspace, int64_t workspace_bytes,
                              hhfm_stream_t stream);
/* Bytes of the workspace of hhfm_fm_bn_fwd_bwd_sqloss for a batch of B samples and K factors; -1 for bad sizes. */
int64_t hhfm_workspace_bytes_fm_bn(int64_t B, int64_t K);
/* The batch-normalised FM forward at evaluation (train_phase=False): the moving statistics, no dropout.
 * out[s] = sum_k (gamma (x - moving_mean) / sqrt(moving_var + eps) + beta) + sum_f b[x_f] + b0, fixed-width rows. */
int hhfm_fm_bn_fwd(const int32_t* col, int64_t B, int64_t F, const float* V, const float* bias, const float* b0, int64_t M,
                   int64_t K, const float* gamma, const float* beta, const float* moving_mean, const float* moving_var,
                   float eps, float* out, hhfm_stream_t stream);
/* Synchronised batch norm (data parallelism): the step of hhfm_fm_bn_fwd_bwd_sqloss on the GLOBAL batch (the ranks'
 * shards concatenated in rank order) as three phases; the caller all-gathers one vector of hhfm_fm_bn_sync_len(K) doubles
 * per rank between them, stacked in rank order ([n_ranks, 2K + 1]).
 *   1. hhfm_fm_bn_sync_stats   the interaction vectors of the local rows -> workspace; stats = this rank's
 *                              (n, mean[K], M2[K]), not finalised.
 *   2. hhfm_fm_bn_sync_loss    stats_all merged in rank order (Chan's formula in double) -> mu, 1/sqrt(var + eps) and the
 *                              moving statistics of the global batch (Bessel correction with the global n); out, the loss
 *                              partials and gb0 (+= local sum g) of the local rows, the dropout mask drawn at each
 *                              sample's GLOBAL index (lower ranks' sizes + local index); sums = (sum g, sum d[K],
 *                              sum d xhat[K]) of the local rows.
 *   3. hhfm_fm_bn_sync_scatter sums_all added in rank order -> dgamma, dbeta (written; the global sums) and the row
 *                              gradients gV / gbias of the local rows, hot rows and touched-row list as in the single call.
 * Every rank derives dgamma, dbeta and the moving statistics from the same gathered vectors in the same order, so they
 * are bit-identical across ranks; gV, gbias, gb0 and the loss partials stay rank-local (the gradient exchange sums them).
 * B may be 0 (the rank still takes part; col, labels and out may then be NULL); when the global batch is empty the layer
 * does not move and dgamma = dbeta = 0.  With n_ranks = 1 the phases reproduce hhfm_fm_bn_fwd_bwd_sqloss bit for bit.
 * The three calls of one step take the same B, K, keep, drop_seed and workspace (hhfm_workspace_bytes_fm_bn_sync(B, K)
 * bytes, 16-byte aligned); per-rank vectors 8-byte aligned. */
int hhfm_fm_bn_sync_stats(const int32_t* col, int64_t B, int64_t F, const float* V, const float* bias, int64_t M, int64_t K,
                          double* stats, void* workspace, int64_t workspace_bytes, hhfm_stream_t stream);
int hhfm_fm_bn_sync_loss(int64_t B, int64_t K, const float* b0, const float* labels, float* out, float* gb0,
                         float* loss_partials, float keep, uint64_t drop_seed, const float* gamma, const float* beta,
                         float* moving_mean, float* moving_var, float eps, float decay, const double* stats_all,
                         int32_t n_ranks, int32_t rank, double* sums, void* workspace, int64_t workspace_bytes,
                         hhfm_stream_t stream);
int hhfm_fm_bn_sync_scatter(const int32_t* col, int64_t B, int64_t F, const float* V, int64_t M, int64_t K, float* gV,
                            float* gbias, int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows, int32_t* touched_count,
                            const int32_t* hot_slot, float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot,
                            int32_t deterministic, float keep, uint64_t drop_seed, float* dgamma, float* dbeta,
                            const double* sums_all, int32_t n_ranks, void* workspace, int64_t workspace_bytes,
                            hhfm_stream_t stream);
/* Doubles in one rank's vector of the synchronised phases (2K + 1); -1 for a bad K. */
int64_t hhfm_fm_bn_sync_len(int64_t K);
/* Bytes of the workspace of the synchronised phases for B local samples and K factors; -1 for bad sizes. */
int64_t hhfm_workspace_bytes_fm_bn_sync(int64_t B, int64_t K);

/* Backward only, for torch.autograd: g = gout[s] given by the caller. */
int hhfm_fm_bwd(const int32_t* row_ptr, const int32_t* col, const float* val, int64_t B, int64_t F,
                const float* V, int64_t M, int64_t K, int32_t interaction, const float* gout,
                float* gV, float* gbias, float* gb0, int32_t deterministic, hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K2  Attentional FM (AFM.py:103-148): pairwise products P_p = E_i*E_j (i<j, lexicographic), attention MLP
 *     Z_p = P_p W + b, s_p = relu(Z_p).p, a = softmax over pairs, afm = sum_p a_p P_p,
 *     out = afm.w_pred + sum_f bias[x_f] + b0;  loss = 0.5*sum(y-out)^2.
 *   idx [B,F] int32 (2 <= F <= 16);  W [K,A] row-major, batt [A], pvec [A], wpred [K];  K, A multiples of 4, <= 128,
 *   in the same 32-tier (reference: A == K).  Gradients accumulate into gV / gbias / gb0 (sort-free scatter, optional
 *   hot-row replicas) and gW [K,A], gbatt [A], gp [A], gwpred [K].  The lamda_attention*||W||^2/2 term (AFM.py:146) is
 *   applied by the caller through hhfm_opt_*_dense_l2 on W.
 * ------------------------------------------------------------------------------------------------ */
int hhfm_afm_fwd(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias, const float* b0,
                 const float* W, const float* batt, const float* pvec, const float* wpred, int64_t M, int64_t K,
                 int64_t A, float* out, hhfm_stream_t stream);
int hhfm_afm_fwd_bwd_sqloss(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias,
                            const float* b0, const float* W, const float* batt, const float* pvec, const float* wpred,
                            int64_t M, int64_t K, int64_t A, const float* labels, float* out, float* gV, float* gbias,
                            float* gb0, float* gW, float* gbatt, float* gp, float* gwpred, float* loss_partials,
                            int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows, int32_t* touched_count,
                            const int32_t* hot_slot, float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot,
                            hhfm_stream_t stream);

/* Training dropout and the attention=0 variant (AFM.py:126,132,134).  The arguments of hhfm_afm_fwd_bwd_sqloss, then:
 *   attention   1: the attention net as above;  0: afm = sum_p P_p = 0.5 (S^2 - sum_f E_f^2) (no attention net; gW, gbatt, gp
 *               are not written)
 *   keep_att, keep_vec   tf.nn.dropout keep probabilities in (0, 1] of the attention weights (per sample and pair; unused
 *               when attention = 0) and of the pooled vector (per sample and column): a_p -> a_p m_p / keep_att and
 *               afm -> afm n / keep_vec with 0/1 masks m = mask(drop_seed, s, p), n = mask(splitmix64(drop_seed), s, k)
 *   sample_base the index of row 0 in the global batch (data parallelism: every rank draws the masks of its own rows), >= 0
 * keep = [1, 1] with attention = 1 runs the kernels of hhfm_afm_fwd_bwd_sqloss unchanged.  hhfm_afm_fwd_attn is the
 * forward (no dropout: the reference evaluates with keep = [1, 1]) for either value of `attention`. */
int hhfm_afm_fwd_bwd_sqloss_dropout(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias,
                                    const float* b0, const float* W, const float* batt, const float* pvec, const float* wpred,
                                    int64_t M, int64_t K, int64_t A, const float* labels, float* out, float* gV, float* gbias,
                                    float* gb0, float* gW, float* gbatt, float* gp, float* gwpred, float* loss_partials,
                                    int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows, int32_t* touched_count,
                                    const int32_t* hot_slot, float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot,
                                    int32_t attention, float keep_att, float keep_vec, uint64_t drop_seed, int64_t sample_base,
                                    hhfm_stream_t stream);
int hhfm_afm_fwd_attn(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* bias, const float* b0,
                      const float* W, const float* batt, const float* pvec, const float* wpred, int64_t M, int64_t K,
                      int64_t A, int32_t attention, float* out, hhfm_stream_t stream);

/* The training pass of K == A == 64, F <= 11 runs as ONE tcgen05 kernel (afm_fused_tc.cu: the three matrix products P W,
 * dZ W^T, P^T dZ as 3xTF32 split products with the operands built in shared memory and the logits / dP in TMEM);
 * hhfm_afm_fwd_bwd_sqloss selects it by shape, HHFM_AFM_TC=0 forces the fp32 CUDA-core kernels. */
/* K2 full-catalog scorer (AFM.py:209-246; afm_topn.cu): scores [C, N] = the AFM forward of every context row with field
 * `item_col` replaced by item n (table row item_base + n), n < N.  Only the F-1 pairs that contain the item are evaluated
 * per (context, item); the context-only pairs are reduced once per context into stats [C, 4] (caller-owned scratch).
 * rows [C, row_stride] int32 (C <= 65535 per call); the entry of column item_col is ignored.  Covered shapes:
 * hhfm_afm_topn_supported(F, K, A) == 1 (K == A in {16, 32, 64}, 2 <= F <= 16); other shapes are scored through
 * hhfm_afm_fwd on expanded rows.  Feed `scores` to hhfm_topn_select for the lists (lowest index first on ties). */
int hhfm_afm_topn_supported(int64_t F, int64_t K, int64_t A);
int hhfm_afm_topn_scores(const int32_t* rows, int64_t row_stride, int64_t C, int64_t F, int32_t item_col, const float* V,
                         const float* bias, const float* b0, const float* W, const float* batt, const float* pvec,
                         const float* wpred, int64_t M, int64_t K, int64_t A, int64_t item_base, int64_t N, float* stats,
                         float* scores, hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K8  DeepFM (DFM.py:104-152): y1_f = feature_bias[x_f], y2 = 0.5((sum e)^2 - sum e^2), a relu MLP tower over the
 *     flattened embeddings, out = [y1 | y2 | H_L] . concat_projection + concat_bias;  loss = 0.5*sum(y-out)^2.
 *   idx [B,F] int32 (F <= 32);  K % 4 == 0;  layer_sizes: HOST array of n_layers (<= 8) widths, last <= 256.
 *   params / gparams: ONE flat buffer, layout
 *     [ layer_0 (F*K x d1) | ... | layer_{L-1} | concat_projection (F+K+d_L) | 0-3 zero pad | bias_0 (d1) | ... | bias_{L-1} | concat_bias ]
 *   (row-major matrices; hhfm_dfm_param_count() elements; the first hhfm_dfm_reg_count() carry DFM.py:145-150's l2).
 *   workspace: hhfm_workspace_bytes_dfm(B, ...) bytes, caller-owned (hidden activations, reused for their gradients).
 *   The GEMMs run on the tensor cores as 3xTF32 splits with fp32 accumulation (dfm_tc.cu; HHFM_DFM_TC=0 selects the fp32
 *   CUDA-core GEMMs, whose layer 0 gathers its A operand straight from V); d(H_0) is scattered into gV by the GEMM epilogue
 *   (optionally through hot-row replicas, as in K1/K3).  workspace: 16-byte aligned.
 *   Gradients ACCUMULATE into gV [M,K], gbias [M], gparams (zero them first).
 * ------------------------------------------------------------------------------------------------ */
int64_t hhfm_dfm_param_count(int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes);
int64_t hhfm_dfm_reg_count(int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes);
int64_t hhfm_workspace_bytes_dfm(int64_t B, int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes);
int hhfm_dfm_fwd(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* feature_bias, int64_t M,
                 int64_t K, const float* params, int32_t n_layers, const int32_t* layer_sizes, float* workspace,
                 float* out, hhfm_stream_t stream);
int hhfm_dfm_fwd_bwd_sqloss(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* feature_bias,
                            int64_t M, int64_t K, const float* params, int32_t n_layers, const int32_t* layer_sizes,
                            const float* labels, float* workspace, float* out, float* gV, float* gbias,
                            float* gparams, float* loss_partials, const int32_t* hot_slot, float* ghot,
                            float* ghot_bias, int32_t n_rep, int32_t n_hot, hhfm_stream_t stream);

/* K8 with the reference's options (mode: hhfm_dfm_mode bits).  The calls above are these with mode 0 (and B_total = B).
 *   NO_FM     out = H_L . proj3 + cbias: no feature_bias gather / gradient (feature_bias and gbias may be NULL), no FM part
 *             of gV; the first F + K projection entries are unused and receive zero gradient.
 *   NO_DEEP   out = [y1 | y2] . proj12 + cbias: no GEMM, no workspace (the queries return 0 bytes; workspace may be NULL),
 *             the layer matrices / biases receive no gradient.  The projection block starts on a multiple of 4 elements
 *             (zero padding after the layer matrices), so [proj_off, reg_count) can be stepped and regularised alone.
 *   LOGLOSS   out = p = sigmoid(logit); loss = tf.losses.log_loss(y, p): sum_s [-y log(p + 1e-7) - (1 - y) log((1 - p) + 1e-7)]
 *             / B_total, d/d logit = p (1 - p) (-y / (p + 1e-7) + (1 - y) / ((1 - p) + 1e-7)) / B_total.  Labels are used
 *             as given.  B_total (>= B) is the batch the mean runs over: the sum of the ranks' B under data parallelism.
 *   Under mse the loss stays 0.5 sum (y - out)^2 and B_total is only checked.  Bad modes fail with HHFM_ERR_BAD_ARG (the
 *   int64 queries return -1); hhfm_last_error() says why.
 *   hhfm_dfm_topn_scores_mode: the same scorer per mode; under LOGLOSS the scores are the sigmoid (the reference ranks by
 *   `out`, so saturated items tie at 1.0f and the lowest index wins in hhfm_topn_select). */
int64_t hhfm_dfm_param_count_mode(int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes, int32_t mode);
int64_t hhfm_dfm_reg_count_mode(int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes, int32_t mode);
int64_t hhfm_workspace_bytes_dfm_mode(int64_t B, int64_t F, int64_t K, int32_t n_layers, const int32_t* layer_sizes,
                                      int32_t mode);
int hhfm_dfm_fwd_mode(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* feature_bias, int64_t M,
                      int64_t K, const float* params, int32_t n_layers, const int32_t* layer_sizes, int32_t mode,
                      float* workspace, float* out, hhfm_stream_t stream);
int hhfm_dfm_fwd_bwd_mode(const int32_t* idx, int64_t B, int64_t F, const float* V, const float* feature_bias, int64_t M,
                          int64_t K, const float* params, int32_t n_layers, const int32_t* layer_sizes, int32_t mode,
                          int64_t B_total, const float* labels, float* workspace, float* out, float* gV, float* gbias,
                          float* gparams, float* loss_partials, const int32_t* hot_slot, float* ghot, float* ghot_bias,
                          int32_t n_rep, int32_t n_hot, hhfm_stream_t stream);

/* K8 full-catalog scorer (DFM.py:219-231): scores [C, N] = the DeepFM forward of every context row with field item_col
 * replaced by item n (table row item_base + n).  The first hidden layer is item-separable, relu((b1 + sum_{f != item}
 * E_f W1_f) + E_n W1_item): its context part is computed once per row and its item part once per item; the remaining layers
 * and the projection run per (row, item) pair (rows s = c*N + n) through the same GEMMs as hhfm_dfm_fwd.  rows [C, row_stride]
 * int32 (column item_col ignored); C*N < 2^31; workspace: hhfm_workspace_bytes_dfm_topn(C, N, ...) bytes, 16-byte aligned.
 * Feed `scores` to hhfm_topn_select for the lists. */
int64_t hhfm_workspace_bytes_dfm_topn(int64_t C, int64_t N, int64_t F, int64_t K, int32_t n_layers,
                                      const int32_t* layer_sizes);
int hhfm_dfm_topn_scores(const int32_t* rows, int64_t row_stride, int64_t C, int64_t F, int32_t item_col, const float* V,
                         const float* feature_bias, int64_t M, int64_t K, const float* params, int32_t n_layers,
                         const int32_t* layer_sizes, int64_t item_base, int64_t N, float* workspace, float* scores,
                         hhfm_stream_t stream);
int64_t hhfm_workspace_bytes_dfm_topn_mode(int64_t C, int64_t N, int64_t F, int64_t K, int32_t n_layers,
                                           const int32_t* layer_sizes, int32_t mode);
int hhfm_dfm_topn_scores_mode(const int32_t* rows, int64_t row_stride, int64_t C, int64_t F, int32_t item_col, const float* V,
                              const float* feature_bias, int64_t M, int64_t K, const float* params, int32_t n_layers,
                              const int32_t* layer_sizes, int32_t mode, int64_t item_base, int64_t N, float* workspace,
                              float* scores, hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K11  Wide&Deep (WDMF.py:51-126: tf.contrib.learn.DNNLinearCombinedClassifier over hashed columns, crossed columns and
 *      128-d embedding columns, DNN [1024, 512, 256]).  The arithmetic of the reference lives inside TensorFlow; this is a
 *      restatement with documented choices (oracle/hhfm_oracle.py wd_*; parity unpinned, SURVEY 8c):
 *   logit = wide(x) + deep(x);  loss = mean sigmoid cross-entropy, labels in {0,1};  probability = sigmoid(logit)
 *   wide(x) = b_wide + sum_f w_lin[x_f] + sum_{i<j} w_cross[p(i,j)][splitmix64((x_i << 32) | x_j) mod n_cross_buckets]
 *             (single columns: one table keyed by the global feature id; pairs p in lexicographic order)
 *   deep(x) = relu MLP over the concatenated embeddings V[x_f] (field order), then a [D_L] -> 1 layer with bias:
 *             the DeepFM tower (K8) with its FM terms off; parameter block = the K8 layout, whose first F + K projection
 *             entries are unused.
 *   hhfm_wd_wide_fwd      out[s] = wide(x_s)
 *   hhfm_wd_deep_fwd      out[s] = extra[s] + deep(x_s)                       (extra = the wide logit, may be NULL)
 *   hhfm_wd_deep_fwd_bwd_logloss   + gV / gparams (accumulated), gsample[s] = d loss / d logit_s, loss partials
 *   hhfm_wd_wide_bwd      g_lin / g_cross / g_b += scatter of gsample
 *   hhfm_opt_ftrl_dense   TF1 ApplyFtrl, learning_rate_power -0.5 (the estimator's optimizer for the wide half)
 * ------------------------------------------------------------------------------------------------ */
int hhfm_wd_wide_fwd(const int32_t* idx, int64_t B, int64_t F, const float* w_lin, const float* w_cross,
                     const float* b_wide, int64_t M, int32_t n_cross_buckets, float* out, hhfm_stream_t stream);
int hhfm_wd_wide_bwd(const int32_t* idx, int64_t B, int64_t F, const float* gsample, int64_t M, int32_t n_cross_buckets,
                     float* g_lin, float* g_cross, float* g_b, hhfm_stream_t stream);
int hhfm_wd_deep_fwd(const int32_t* idx, int64_t B, int64_t F, const float* V, int64_t M, int64_t K, const float* params,
                     int32_t n_layers, const int32_t* layer_sizes, const float* extra, float* workspace, float* out,
                     hhfm_stream_t stream);
int hhfm_wd_deep_fwd_bwd_logloss(const int32_t* idx, int64_t B, int64_t F, const float* V, int64_t M, int64_t K,
                                 const float* params, int32_t n_layers, const int32_t* layer_sizes, const float* labels,
                                 const float* extra, float* workspace, float* out, float* gV, float* gparams,
                                 float* gsample, float* loss_partials, const int32_t* hot_slot, float* ghot, int32_t n_rep,
                                 int32_t n_hot, hhfm_stream_t stream);
int hhfm_opt_ftrl_dense(float* w, float* accum, float* linear, float* g, int64_t n, float lr, float l1, float l2,
                        int32_t zero_grad, hhfm_stream_t stream);

/* fp32-accurate GEMM on the tensor cores (the building block of the DeepFM tower, dfm_tc.cu): C[M,N] = A[M,K] . B[N,K]^T,
 * row-major operands with K contiguous, 3xTF32 split (A_hi.B_hi + A_hi.B_lo + A_lo.B_hi) with fp32 accumulation in TMEM.
 * lda / ldb / ldc are multiples of 4 floats, pointers 16-byte aligned; workspace: (M*lda + N*ldb) floats. */
int hhfm_gemm_tn_tf32x3(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int64_t N, int64_t K, float* C,
                        int64_t ldc, float* workspace, hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K3  HHFM (OurModel7.py:105-184) and BPR (BPR.py:76-88) pairwise ranking
 * Record layout (int32, row stride `stride` >= 2+n_ctx+n_time+n_neg, stride % 4 == 0, 16-byte aligned):
 *   [user, item+, ctx_0..ctx_{n_ctx-1}, time_0..time_{n_time-1}, neg_0..neg_{n_neg-1}, pad...]
 *   hyb = Pool_stack(stack[V[user], Pool_ctx(V[ctx]), Pool_time(V[time])]);  BPR: n_ctx = n_time = 0
 *   pos = hyb.V[item+]; neg_j = hyb.V[neg_j]; loss = -sum log(sigmoid(pos - max_j neg_j))
 *   reduce_max backward splits equally among tied maxima (TF semantics).
 * ------------------------------------------------------------------------------------------------ */
int hhfm_pairrank_fwd(const int32_t* idx, int64_t B, int64_t stride, int32_t n_ctx, int32_t n_time, int32_t n_neg,
                      int32_t pool_ctx, int32_t pool_time, int32_t pool_stack, const float* V, int64_t M, int64_t K,
                      float* pos_out, float* neg_out, hhfm_stream_t stream);

int hhfm_pairrank_fwd_bwd(const int32_t* idx, int64_t B, int64_t stride, int32_t n_ctx, int32_t n_time,
                          int32_t n_neg, int32_t pool_ctx, int32_t pool_time, int32_t pool_stack, const float* V,
                          int64_t M, int64_t K, float* pos_out, float* neg_out, float* gV, float* loss_partials,
                          int32_t* touch_stamp, int32_t stamp, int32_t* touched_rows, int32_t* touched_count,
                          const int32_t* hot_slot, float* ghot, int32_t n_rep, int32_t n_hot,
                          int32_t deterministic, hhfm_stream_t stream);

/* Pooled context groups of the sum-pooling training pass.  With every pool mode HHFM_POOL_SUM only the sum of the pooled
 * rows enters the model, so pooled columns with small vocabularies can be pre-pooled: the columns of a group (id ranges
 * [col_lo[c], col_lo[c] + col_card[c]), disjoint, inside [0, M)) are replaced by one row of the group table
 *   S_g[k] = sum over the members c, in record order, of V[col_lo[c] + d_c(k)],
 * k = sum_c d_c * prod_{c' before c} col_card[c'] (mixed radix, first member least significant), and the gradient of that
 * row is handed back to the member rows after the pass.  Per positive this gathers and reduces one row per group instead
 * of one per column.
 *   hhfm_pool_groups_attach registers the plan under the table pointer V (col_group[c]: group number of pooled column c,
 *     c < n_pool = n_ctx + n_time, or -1 = ungrouped) and allocates S and G ([rows, K] each, G zero).  A later plan for
 *     the same V replaces it.  *handle identifies the plan for detach.
 *   hhfm_pairrank_fwd_bwd then runs, on the caller's stream: the pre-sum of S, the grouped training kernel, the
 *     expansion of G into gV (fixed summation order) and the clearing of G.  The plan is used when M, K, n_ctx + n_time,
 *     stride and the current device match it, every pool mode is HHFM_POOL_SUM, n_neg == 10, K in {32, 64, 128},
 *     deterministic == 0 and no touched-row tracking or positive / negative outputs are requested,
 *     and the large-table (staged) kernel does not run; otherwise the call is the ungrouped one.  A sample whose member
 *     id lies outside the planned range pools and scatters that group's member rows individually (hot-row plan / gV).
 *     Member rows should not be hot rows: nothing but those fallback samples should reduce into them during the pass.
 *     HHFM_POOL_GROUPS=0 ignores every plan.
 *   hhfm_pool_groups_detach removes the plan (no-op unless V and handle match).
 *   hhfm_pool_groups_tables returns the plan's S, G and their row count. */
int hhfm_pool_groups_attach(const float* V, int64_t M, int64_t K, int32_t n_pool, int64_t stride, const int32_t* col_group,
                            const int32_t* col_lo, const int32_t* col_card, int64_t* handle);
int hhfm_pool_groups_detach(const float* V, int64_t handle);
int hhfm_pool_groups_tables(const float* V, float** S, float** G, int64_t* rows);

/* Backward only, for torch.autograd: dpos [B], dneg [B,n_neg] (nullable) given by the caller. */
int hhfm_pairrank_bwd(const int32_t* idx, int64_t B, int64_t stride, int32_t n_ctx, int32_t n_time, int32_t n_neg,
                      int32_t pool_ctx, int32_t pool_time, int32_t pool_stack, const float* V, int64_t M, int64_t K,
                      const float* dpos, const float* dneg, float* gV, int32_t deterministic, hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K4  generic segmented scatter-add of rows: dst[rows[i], :] += src[i, :]   (TF UnsortedSegmentSum /
 * IndexedSlices aggregation implicit in every `.minimize`, FM.py:132).  Sort-free: vector reductions.
 * ------------------------------------------------------------------------------------------------ */
int hhfm_scatter_add_rows(const int32_t* rows, const float* src, int64_t n, int64_t K, float* dst, int64_t M,
                          hhfm_stream_t stream);

/* Coalesced-sparse gradient exchange (SURVEY 8e; data-parallel training of tables too large for a dense all-reduce):
 *   hhfm_gather_rows  out[i, :] = table[ids[i], :] (K == 1 or K % 4 == 0); zero_src != 0 clears the source rows, so that the
 *                     ranks' row lists (own one included) can be added back in rank order -> bit-identical replicas;
 *   hhfm_touch_rows   appends ids not yet stamped in this step to the touched-row list the *_rows optimizers consume. */
int hhfm_gather_rows(float* table, const int32_t* ids, int64_t n, int64_t K, int64_t M, float* out, int32_t zero_src,
                     hhfm_stream_t stream);
int hhfm_touch_rows(const int32_t* ids, int64_t n, int32_t* stamp_arr, int32_t stamp, int32_t* rows, int32_t* count,
                    hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K5  optimizers with TF-1.x semantics (FM.py:129-136; BPR.py:93 / MF.py:104 use acc0 = 1e-8)
 *   adagrad : acc += g^2; w -= lr*g/sqrt(acc)                (no epsilon)
 *   adam    : lr_t = lr*sqrt(1-b2^t)/(1-b1^t) is computed by the CALLER and passed as `lr`;
 *             m = b1*m+(1-b1)*g; v = b2*v+(1-b2)*g^2; w -= lr*m/(sqrt(v)+eps)
 *   momentum: acc = acc*mu + g; w -= lr*acc
 *   sgd     : w -= lr*g
 * _dense_l2: g_eff = g + lamda*w over all n elements (the reference's l2_regularizer on the embedding table
 *   makes the gradient dense, FM.py:124).  sq_partials (nullable, [hhfm_partials_len()]) receives per-CTA
 *   partial sums of w^2 BEFORE the update, for the regulariser term of the reported loss.
 * _rows: only the listed rows move (TF SparseApply*): rows int32[*n_rows_dev], each row has K elements.
 *   zero_grad = 1 clears the consumed gradient entries so the buffer is ready for the next step.
 * ------------------------------------------------------------------------------------------------ */
int hhfm_opt_adagrad_dense_l2(float* w, float* acc, float* g, int64_t n, float lr, float lamda, int32_t zero_grad,
                              float* sq_partials, hhfm_stream_t stream);
int hhfm_opt_adam_dense_l2(float* w, float* m, float* v, float* g, int64_t n, float lr_t, float beta1, float beta2,
                           float eps, float lamda, int32_t zero_grad, float* sq_partials, hhfm_stream_t stream);
int hhfm_opt_momentum_dense_l2(float* w, float* acc, float* g, int64_t n, float lr, float momentum, float lamda,
                               int32_t zero_grad, float* sq_partials, hhfm_stream_t stream);
int hhfm_opt_sgd_dense_l2(float* w, float* g, int64_t n, float lr, float lamda, int32_t zero_grad,
                          float* sq_partials, hhfm_stream_t stream);
int hhfm_opt_adagrad_rows(float* w, float* acc, float* g, const int32_t* rows, const int32_t* n_rows_dev,
                          int64_t max_rows, int64_t K, float lr, int32_t zero_grad, hhfm_stream_t stream);
int hhfm_opt_momentum_rows(float* w, float* acc, float* g, const int32_t* rows, const int32_t* n_rows_dev,
                           int64_t max_rows, int64_t K, float lr, float momentum, int32_t zero_grad,
                           hhfm_stream_t stream);
int hhfm_opt_sgd_rows(float* w, float* g, const int32_t* rows, const int32_t* n_rows_dev, int64_t max_rows,
                      int64_t K, float lr, int32_t zero_grad, hhfm_stream_t stream);

/* Lazy-exact dense L2 (SURVEY.md 7, hard part 2-ii): the reference's l2_regularizer on the table (FM.py:124,
 * OurModel7.py:181-182) moves every row every step (g = lamda*w for an untouched row).  Those steps depend on the row alone,
 * so they are replayed -- same fp32 operations, same order, bit-identical to hhfm_opt_adagrad_dense_l2 -- when the row is next
 * gathered and at flush.  last_step [M] int32 = the optimizer step each row reflects.
 *   hhfm_mark_rows: rows [*count] = the distinct ids >= 0 among ids[0, n) (stamp stores + compaction; stamp as in K1).
 *   hhfm_opt_adagrad_l2_replay: replays steps last_step[row]+1 .. upto for the listed rows (rows == NULL: all M rows) and
 *     sets last_step = upto.
 *   hhfm_opt_adagrad_rows_l2: step `step` on the listed rows with g_eff = g + lamda*w; sets last_step = step. */
int hhfm_mark_rows(const int32_t* ids, int64_t n, int32_t* stamp_arr, int32_t stamp, int64_t M, int32_t* rows, int32_t* count,
                   hhfm_stream_t stream);
/* hhfm_touched_compact: rows[0, *count) = the rows r < M with stamp_arr[r] == stamp (any order; *count is cleared first).
 *   Under data parallelism with Momentum the ranks' stamp arrays are MAX all-reduced (one int32 per row) and compacted
 *   here: the list is then the union of the rows touched on any rank, which SparseApplyMomentum (K5 *_rows) consumes. */
int hhfm_touched_compact(const int32_t* stamp_arr, int32_t stamp, int64_t M, int32_t* rows, int32_t* count,
                         hhfm_stream_t stream);
int hhfm_opt_adagrad_l2_replay(float* w, float* acc, int32_t* last_step, const int32_t* rows, const int32_t* n_rows_dev,
                               int64_t max_rows, int64_t M, int64_t K, float lr, float lamda, int32_t upto, hhfm_stream_t stream);
int hhfm_opt_adagrad_rows_l2(float* w, float* acc, float* g, const int32_t* rows, const int32_t* n_rows_dev, int64_t max_rows,
                             int64_t K, float lr, float lamda, int32_t zero_grad, int32_t* last_step, int32_t step,
                             hhfm_stream_t stream);

/* gV[hot_rows[s], :] += sum_r ghot[r, s, :] (and gbias likewise), replicas cleared; fixed summation order. */
int hhfm_hot_fold(float* ghot, float* ghot_bias, int32_t n_rep, int32_t n_hot, int64_t K, const int32_t* hot_rows,
                  float* gV, float* gbias, hhfm_stream_t stream);

/* loss_out[0] = sum(loss_partials) + half_lamda * sum(sq_partials)   (fixed summation order; sq may be NULL) */
int hhfm_loss_finalize(const float* loss_partials, const float* sq_partials, float half_lamda, float* loss_out,
                       hhfm_stream_t stream);

/* Measurement aid: stream `n_floats` floats `iters` times with L1-bypassing 16-byte loads (an L2-resident buffer gives the
 * L2 -> SM read bandwidth that bench.py quotes as the peak of the L2-bound gather kernels). */
int hhfm_l2_read_sweep(const float* buf, int64_t n_floats, int32_t iters, float* sink, hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K12  data-parallel training step (p2p.cu; SURVEY.md 8e): hot-replica fold + cross-GPU all-reduce of the gradient arena
 *   + TF1 optimizer + loss reduction in ONE persistent cooperative kernel.  The reference has no distributed code; this
 *   replaces what `optimizer.minimize` (FM.py:129-136, OurModel7.py:185-189) does after the gradients exist, for a batch
 *   whose rows are sharded across the GPUs of one box.
 *
 *   arena        rank-private gradient buffer; floats [0, n_grad) are consumed (and cleared); the table gradient [M, K]
 *                occupies [0, M*K).
 *   segs         up to 4 variables whose gradients are arena[offset, offset+n): w / s1 / s2 as in K5, lamda per segment
 *                (g_eff = g + lamda*w; the loss gets 0.5*lamda*sum(w^2) of the weights BEFORE the update).
 *   ghot...      the two-level scatter plan of K1/K3 (NULL / 0 = none): hot_slot [M] as given to the scatter kernels,
 *                bias_off = offset of the feature_bias gradient (with ghot_bias).
 *   x_local      this rank's exchange buffer, hhfm_dp_exchange_floats(n_grad) floats.  For n_ranks > 1 it must be symmetric
 *                memory: x_peers_host[r] = address of rank r's buffer in THIS process (own one included), x_multicast =
 *                the multicast alias of the same buffers (multimem.ld_reduce / multimem.st) or NULL (peer loads / stores).
 *   flag_peers_host[r]  address of rank r's flag array (hhfm_dp_flag_ints() int32, zero-initialised, symmetric memory).
 *   state        device int32[4], zero-initialised: [0] step counter, [2] ticket (both owned by the kernel), [1] sticky
 *                error flag -- set when a cross-GPU flag wait took longer than timeout_s (<= 0: 120 s); later steps return
 *                at once, the host reads it back with the loss.  No trap: the CUDA context stays usable.
 *   reg_workspace  >= 257 floats.   loss_out[0] = sum over ranks of sum(loss_partials) + regulariser.
 *   Adam: `lr` is lr_t (K5); Momentum: beta1 carries the momentum.  All replicas consume the same reduced bits, so they
 *   stay bit-identical.  n_ranks == 1: fold + optimizer + loss of a single-GPU step in one launch.
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
  float* w;
  float* s1;
  float* s2;
  int64_t offset;
  int64_t n;
  float lamda;
  int32_t reserved;
} hhfm_dp_segment;
int64_t hhfm_dp_exchange_floats(int64_t n_grad);
int64_t hhfm_dp_flag_ints(void);
int hhfm_dp_step(int32_t kind, const hhfm_dp_segment* segs, int32_t n_segs, float* arena, int64_t n_grad, float* ghot,
                 float* ghot_bias, int32_t n_rep, int32_t n_hot, int64_t K, int64_t M, const int32_t* hot_slot, int64_t bias_off,
                 const float* loss_partials, float* x_local, float* x_multicast, const int64_t* x_peers_host,
                 const int64_t* flag_peers_host, int32_t rank, int32_t n_ranks, int32_t* state, float lr, float beta1,
                 float beta2, float eps, float* reg_workspace, float* loss_out, double timeout_s, hhfm_stream_t stream);
/* hhfm_dp_step_touched: hhfm_dp_step with IndexedSlices variables (TF1 SparseApply*: only the rows touched on SOME rank
 *   move; a touched row whose summed gradient is 0 still takes the step, e.g. Momentum's accum decays).  seg_widths (host,
 *   n_segs): row width of each segment, 0 = dense as in hhfm_dp_step; a segment with a width w covers rows [0, n / w) of
 *   the table (n / w <= M, lamda 0).  stamps [M] / stamp: this rank's touched-row stamps from the scatter kernels (K1).
 *   Each rank's touched bits travel with its gradient and are OR-reduced with it, so every replica makes the same
 *   decision; with n_ranks == 1 the local stamps decide.  x_local then holds hhfm_dp_exchange_floats_touched(n_grad)
 *   floats.  Other arguments as hhfm_dp_step; any optimizer kind. */
int64_t hhfm_dp_exchange_floats_touched(int64_t n_grad);
int hhfm_dp_step_touched(int32_t kind, const hhfm_dp_segment* segs, int32_t n_segs, const int32_t* seg_widths,
                         const int32_t* stamps, int32_t stamp, float* arena, int64_t n_grad, float* ghot, float* ghot_bias,
                         int32_t n_rep, int32_t n_hot, int64_t K, int64_t M, const int32_t* hot_slot, int64_t bias_off,
                         const float* loss_partials, float* x_local, float* x_multicast, const int64_t* x_peers_host,
                         const int64_t* flag_peers_host, int32_t rank, int32_t n_ranks, int32_t* state, float lr,
                         float beta1, float beta2, float eps, float* reg_workspace, float* loss_out, double timeout_s,
                         hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K10  CARS2 (CARS2.py:66-187), the context-aware baseline of main.py:50-63.
 *   params / gparams: ONE flat block [ UI (n_ui x D) | Context (M x Dc) | W (D x Dp x Dc) | Z (D x Dq x Dc) | A (Dp) | B (Dq) ],
 *   hhfm_cars2_param_count() floats, all of it L2-regularised (CARS2.py:116-123: apply hhfm_opt_*_dense_l2 to the block).
 *   hhfm_cars2_fwd: mode 0 -> out[B] = PositiveFeadback of records [user, item, fea]; mode 2 -> out[B, D] = u + T c, the
 *   query vector whose dot product with the item rows ranks the catalog (CARS2.topk, :171-187).
 *   hhfm_cars2_fwd_bwd: records [user, item, fea, neg...]; loss partials of -sum log sigmoid(Pos - Neg); gradients ACCUMULATE.
 *   workspace: hhfm_workspace_bytes_cars2(B, D, Dc) bytes.  D, Dc <= 128.
 * ------------------------------------------------------------------------------------------------ */
int64_t hhfm_cars2_param_count(int64_t n_ui, int64_t M, int64_t D, int64_t Dp, int64_t Dq, int64_t Dc);
int64_t hhfm_workspace_bytes_cars2(int64_t B, int64_t D, int64_t Dc);
int hhfm_cars2_fwd(const int32_t* rec, int64_t B, int64_t stride, const float* params, int64_t n_ui, int64_t M, int64_t D,
                   int64_t Dp, int64_t Dq, int64_t Dc, int32_t mode, float* out, float* workspace, hhfm_stream_t stream);
int hhfm_cars2_fwd_bwd(const int32_t* rec, int64_t B, int64_t stride, int32_t n_neg, const float* params, int64_t n_ui,
                       int64_t M, int64_t D, int64_t Dp, int64_t Dq, int64_t Dc, float* gparams, float* loss_partials,
                       float* workspace, hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K9  device negative sampler and evaluate_AUC (sampler.cu; SURVEY.md 8f-1, 8f-2)
 * hhfm_sample_negatives: out[r, out_col0 + j] (row stride out_stride) = a uniform item id in [n_user, n_user+n_item),
 *   re-drawn while key_id[r]*span + item is in the sorted int64 list pf_codes (= `item in positive_feedback[key(row)]`,
 *   FM.py:284-294); key_id[r] < 0 (key never trained) or key_id == NULL rejects nothing.  Every draw is
 *   splitmix64(seed, cell = r*num + j, attempt): reproducible and order independent (oracle: sample_negative_hashed).
 * hhfm_expand_rows: out[(r*num + j), :F] = rows[r, :F] with column 1 replaced by items[r*num + j], columns [F, out_stride)
 *   = -1 (FM.py:303-305).
 * hhfm_auc_count: *wins += #{(r, j): pos[r] > neg[r*num + j]}                                        (FM.py:321-323).
 * ------------------------------------------------------------------------------------------------ */
int hhfm_sample_negatives(const int32_t* key_id, int64_t n, int32_t num, int32_t n_user, int32_t n_item,
                          const int64_t* pf_codes, int64_t n_codes, int64_t span, uint64_t seed, int32_t* out,
                          int64_t out_stride, int64_t out_col0, hhfm_stream_t stream);
int hhfm_expand_rows(const int32_t* rows, int64_t n, int32_t F, int64_t stride, const int32_t* items, int32_t num,
                     int32_t* out, int32_t out_stride, hhfm_stream_t stream);
int hhfm_auc_count(const float* pos, const float* neg, int64_t n, int32_t num, uint64_t* wins, hhfm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K6  full-catalog top-N (FM.py:172-185, BPR.py:131-136, MF.py:144-149, OurModel7.py:229-295)
 * Exact path (bit-identical to the oracle's canonical fp32 order: k ascending, separately rounded mul/add):
 *   build_query -> score_exact -> select.
 *   A: int32 [C, stride] rows [user, item, ctx..., time...] (the reference's `feed_dict` rows, FM.py:333).
 *   items = V + n_user*K (the item id range is contiguous, FM.py:175); item_bias = bias + n_user or NULL.
 *   FM: score = fl(bias_n + sum_k fl(q_k * fl(v_nk + Fc_k)));  others: score = sum_k fl(q_k*v_nk).
 * select: per row the tp best of `n` (score, id) pairs under (score desc, id asc) == tf.nn.top_k order.
 *   ids == NULL means id = column index; counts == NULL means every row has n entries.  Output ids get
 *   id_offset added (item-shard offset for the multi-GPU merge).  tp <= 1024.
 * ------------------------------------------------------------------------------------------------ */
int hhfm_topn_build_query(int32_t kind, const int32_t* A, int64_t C, int64_t stride, int32_t n_ctx, int32_t n_time,
                          int32_t pool_ctx, int32_t pool_time, int32_t pool_stack, const float* V, int64_t M,
                          int64_t K, float* Q, float* Fc, hhfm_stream_t stream);
int hhfm_topn_score_exact(int32_t kind, const float* Q, const float* Fc, int64_t C, const float* items,
                          const float* item_bias, int64_t N, int64_t K, float* scores, int64_t score_stride,
                          hhfm_stream_t stream);
int hhfm_topn_select(const float* scores, const int32_t* ids, const int32_t* counts, int64_t C, int64_t row_stride,
                     int64_t n, int32_t tp, int32_t id_offset, float* out_scores, int32_t* out_ids,
                     hhfm_stream_t stream);

/* Tensor-core path (topn_tc.cu): the same top-N lists, bit-identical, with the catalog scoring done as a bf16 GEMM
 * on tcgen05 (TMA-staged operands, fp32 accumulators in TMEM) used as a FILTER, then exact fp32 rescoring:
 *   hhfm_topn_tc_prepare_items  items fp32 [N,K] (+bias) -> bf16 operand [N,Kp] and stats = {max ||v||, max |b|}
 *                               (cache it while the weights do not change; size from hhfm_topn_tc_item_operand_bytes)
 *   hhfm_topn_score             queries -> bf16; GEMM #1 with a fused group-max epilogue; tau_c = tp-th largest group
 *                               maximum; GEMM #2 whose epilogue emits the ids with approx score >= tau_c - 2E_c;
 *                               survivors stay in `workspace`
 *   hhfm_topn_rescore_merge     survivors are rescored exactly (canonical order) and selected under
 *                               (score desc, id asc); id_offset = item-shard offset (multi-GPU merge).
 *                               overflow[c] = 1 marks a row whose candidate buffer overflowed (tie-degenerate data):
 *                               the caller must redo that row with the exact path.
 * hhfm_topn_tc_supported says whether (kind, N, K, tp) is covered (K + bias chunk <= 256, ceil(N/32) >= tp).
 * workspace: 256-byte aligned, hhfm_workspace_bytes_topn bytes; item_operand: 128-byte aligned. */
int hhfm_topn_tc_supported(int32_t kind, int64_t N, int64_t K, int32_t tp);
int64_t hhfm_topn_tc_item_operand_bytes(int32_t kind, int64_t N, int64_t K);
int64_t hhfm_workspace_bytes_topn(int32_t kind, int64_t C, int64_t N, int64_t K, int32_t tp);
int hhfm_topn_tc_prepare_items(int32_t kind, const float* items, const float* item_bias, int64_t N, int64_t K,
                               void* item_operand, float* stats, hhfm_stream_t stream);
int hhfm_topn_score(int32_t kind, const float* Q, const float* Fc, int64_t C, const void* item_operand, int64_t N,
                    int64_t K, int32_t tp, const float* stats, void* workspace, int64_t workspace_bytes,
                    hhfm_stream_t stream);
int hhfm_topn_rescore_merge(int32_t kind, const float* Q, const float* Fc, int64_t C, const float* items,
                            const float* item_bias, int64_t N, int64_t K, int32_t tp, int32_t id_offset,
                            void* workspace, int64_t workspace_bytes, float* out_scores, int32_t* out_ids,
                            int32_t* overflow, hhfm_stream_t stream);

/* K7  evaluate_TopK walk (FM.py:336-357) including its positive_feedback quirk.
 *   pred [C,tp] GLOBAL item ids; target [C]; target_in_pf [C] = (item in positive_feedback[key]) computed
 *   by the host.  rank_code[c] = n >= 0: hit at counter n;  -1: miss (appends 0);  -2: row appends nothing. */
int hhfm_metrics_walk(const int32_t* pred, const int32_t* target, const uint8_t* target_in_pf, int64_t C,
                      int32_t tp, int32_t TopK, int32_t* rank_code, hhfm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* HHFM_SM100_H */
