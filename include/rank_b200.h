/*
 * rank_b200.h — C ABI of librank_b200.so: the B200 (sm_100a) CTR hot path.
 *
 * The reference (reallinshengxiang/Implementation-of-Rank-Algorithm-for-Mainstream-
 * Recommender-Systems) has no FFI of its own: its hot path is the body of each
 * nn.Module.forward plus the autograd backward of it.  Every entry point below replaces one
 * such body (cited as file:line relative to the reference root, algorithm/...).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the comment says "host";
 *   - tables are fp32 row-major [rows, dim]; indices are int64 (torch.long), lengths int64;
 *   - all work is enqueued on `stream`; the library never synchronises, allocates or frees
 *     device memory, so a whole training step is CUDA-graph capturable;
 *   - return value: 0 = ok, >0 = cudaError_t of the failing runtime call, <0 = argument
 *     error; rk_last_error() gives a thread-local message;
 *   - out-of-range indices are clamped to row 0 and raise bit 0 of *err_flag (the reference
 *     raises IndexError on CPU / device-asserts on CUDA); err_flag may be NULL.
 */
#ifndef RANK_B200_H
#define RANK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RK_ABI_VERSION 3
#define RK_MAX_FIELDS 24
#define RK_MAX_TABLES 32
#define RK_MAX_LAYERS 8

typedef void* rk_stream_t; /* cudaStream_t */

/* One sparse field: a table and the index column that reads it (nn.Embedding + lookup,
 * e.g. DeepFM/deepfm.py:90-98,123-132; DCN/dcn.py:130-137,163-167). */
typedef struct rk_field {
    const float*   weight;  /* [rows, dim] */
    const int64_t* idx;     /* [n] */
    int64_t        rows;    /* V */
    int32_t        dim;     /* D */
    int32_t        out_off; /* first column of this field in the concatenated row */
} rk_field_t;

/* One table's share of the embedding-gradient reduction: per-occurrence gradient rows live at
 * g + occurrence*ld (+0..dim-1); the dense gradient [rows, dim] is written to dw. */
typedef struct rk_grad_table {
    const float* g;
    int64_t      ld;
    float*       dw;     /* [rows, dim], must be zero-filled by the caller */
    int32_t      dim;
    int32_t      field;  /* which field's (sorted) occurrences feed this table */
} rk_grad_table_t;

int         rk_version(void);
const char* rk_last_error(void);
int         rk_device_sm_count(void);
/* Measurement aid (bench.py): occupy `stream` for `us` microseconds (<= 100 ms) so the host can
 * queue a step behind it and CUDA events around each call then see device time only. */
int         rk_debug_spin(int us, rk_stream_t stream);
long long   rk_launch_count(void);   /* kernels launched through this library so far (process-wide) */

/* ---- sparse embedding-gradient reduction (autograd of nn.Embedding: embedding_dense_backward,
 *      reached from loss.backward() e.g. DIN/din.py:346) -------------------------------------
 * rk_plan_build sorts all occurrences of F index columns by (field, row), stably, so that the
 * later reduction sums each row's gradients in occurrence order: deterministic, no atomics.
 *   idx[f]  device pointer to n[f] int64 indices, rows[f] = table height      (host arrays)
 *   sorted_keys[n_total], perm[n_total] : outputs (uint32); perm holds the occurrence number
 *   inside its field.  ws: scratch of rk_plan_workspace_bytes(n_total).
 *   Sequence fields may drop padded positions, whose gradient is identically zero, from the
 *   reduction: live_mode[f] = RK_LIVE_PREFIX keeps t < seq_len[f][b] of every sample b (n[f] =
 *   B*seq_T[f]); RK_LIVE_PREFIX_OR_EMPTY also keeps every t of samples with length 0 (DIN's
 *   softmax mode gives those uniform weights).  seq_len/seq_T/live_mode may be NULL (all live). */
#define RK_LIVE_ALL 0
#define RK_LIVE_PREFIX 1
#define RK_LIVE_PREFIX_OR_EMPTY 2
size_t rk_plan_workspace_bytes(int64_t n_total);
int rk_plan_build(const int64_t* const* idx, const int64_t* n, const int64_t* rows, int F,
                  const int64_t* const* seq_len, const int32_t* seq_T, const int32_t* live_mode,
                  uint32_t* sorted_keys, uint32_t* perm, void* ws, size_t ws_bytes,
                  int32_t* err_flag, rk_stream_t stream);
/* ws for the reduction: rk_reduce_workspace_bytes(sum over tables of ceil(n/16)*dim floats). */
size_t rk_reduce_workspace_bytes(const int64_t* n, int F, const rk_grad_table_t* tables,
                                 int n_tables);
int rk_embgrad_segment_reduce(const uint32_t* sorted_keys, const uint32_t* perm,
                              const int64_t* n, const int64_t* rows, int F,
                              const rk_grad_table_t* tables, int n_tables, void* ws,
                              size_t ws_bytes, rk_stream_t stream);

/* One-launch reduction for per-sample index columns (n <= RK_DIRECT_MAX_N occurrences per table; every
 * per-sample field at batch <= 8192), replacing rk_plan_build + a memset + rk_embgrad_segment_reduce for
 * those tables (same reference code: embedding_dense_backward under loss.backward(), e.g. DCN/dcn.py:166).
 * Output-partitioned: every CTA owns 256 rows of one table, scans the whole index column, orders the
 * occurrences that fall into its rows by (row, occurrence) and sums their gradient rows in that order
 * (runs longer than 32 occurrences: fixed interleaved slots + a fixed tree).  dw is written completely —
 * zeros for rows no occurrence touches — so it need NOT be pre-zeroed.  Tables of one launch that share
 * idx, rows and n (DeepFM / FwFM: the [rows,1] and [rows,D] tables of a field) share the scan and the order.
 * Deterministic, no float atomics.  Out-of-range indices count as row 0 and raise *err_flag. */
#define RK_DIRECT_MAX_N 8192
typedef struct rk_direct_table {
    const int64_t* idx;   /* [n] index column */
    const float*   g;     /* gradient row of occurrence o at g + o*ld (+0..dim-1) */
    int64_t        ld;
    float*         dw;    /* [rows, dim], written completely */
    int64_t        rows;
    int64_t        n;
    int32_t        dim;
    int32_t        reserved;
} rk_direct_table_t;
int rk_embgrad_direct_reduce(const rk_direct_table_t* tables, int n_tables, int32_t* err_flag,
                             rk_stream_t stream);

/* ---- gather + concat (the per-field lookup loops + torch.cat, DCN/dcn.py:163-169,
 *      DeepCrossing/deepcrossing.py:148-155) ------------------------------------------------
 * out[b, 0:n_dense] = dense[b, :]; out[b, off_f:off_f+dim_f] = W_f[idx_f[b], :]. */
int rk_gather_concat_fwd(const rk_field_t* fields, int F, const float* dense, int n_dense,
                         int64_t B, float* out, int ld_out, int32_t* err_flag,
                         rk_stream_t stream);

/* ---- DeepFM FM part (DeepFM/deepfm.py:121-142) ------------------------------------------
 * second[f] are the F second-order tables (dim D each, idx shared with first[f], dim 1).
 * deep_input[B, F*D] = cat_f e_f; fm_first[B] = sum_f w_f; fm_second[B] = 0.5*sum_d((sum_f e)^2
 * - sum_f e^2). */
int rk_deepfm_fwd(const rk_field_t* second, const float* const* first_weight, int F, int64_t B,
                  float* deep_input, float* fm_first, float* fm_second, int32_t* err_flag,
                  rk_stream_t stream);
/* Per-occurrence second-order gradients g_rows[B, F*D] = g_deep + g_second*(S - e_f);
 * g_deep or g_second may be NULL (treated as zero). */
int rk_deepfm_bwd(const float* deep_input, const float* g_deep, const float* g_second, int F,
                  int D, int64_t B, float* g_rows, rk_stream_t stream);

/* ---- FwFM (FwFM/fwfm.py:87-139; "next" row of the scope table) -----------------------------
 * second[f]: the F embedding tables (dim D each); first_weight[f]: the `linear` tables [rows,1],
 * same idx; field_weight[P], P = F(F-1)/2 in the reference's pair order (i outer, j inner,
 * fwfm.py:126-135); bias[1].  emb[B, F*D] = cat_f e_f (kept for the backward);
 * y[B] = sigmoid(sum_f w_f + sum_p r_p <e_i, e_j> + bias)  (fwfm.py:137-139). */
int rk_fwfm_fwd(const rk_field_t* second, const float* const* first_weight,
                const float* field_weight, const float* bias, int F, int64_t B, float* emb,
                float* y, int32_t* err_flag, rk_stream_t stream);
/* Rows of `partials` the backward may use (one per CTA). */
int rk_fwfm_bwd_ctas(void);
/* g_z[B] = g_y * y * (1-y) (the per-occurrence gradient of every first-order table);
 * g_rows[B, F*D]: per-occurrence gradients of the embedding rows;
 * g_pair[P+1] = [d field_weight (P), d bias]; partials: scratch [rk_fwfm_bwd_ctas()][P+1].
 * Sums over the batch have a fixed order (no float atomics). */
int rk_fwfm_bwd(const float* emb, const float* y, const float* g_y, const float* field_weight,
                int F, int D, int64_t B, float* g_rows, float* g_z, float* partials,
                float* g_pair, rk_stream_t stream);

/* ---- DCN CrossNet (cross_layer + loop, DCN/dcn.py:25-50,169-173) -------------------------
 * fwd: x0 = [dense | gathered rows] -> concat_all[B,d]; x_{l+1} = x0*(x_l.w_l) + b_l + x_l
 * -> cross_vec[B,d].  w, b: [L, d]. */
int rk_crossnet_fwd(const rk_field_t* fields, int F, const float* dense, int n_dense,
                    const float* w, const float* b, int L, int64_t B, float* concat_all,
                    float* cross_vec, int32_t* err_flag, rk_stream_t stream);
/* bwd: g_x0[B,d] = g_concat_all + d(cross_vec)/d(x0) . g_cross_vec (either may be NULL). */
int rk_crossnet_bwd(const float* concat_all, const float* w, const float* b, int L, int d,
                    int64_t B, const float* g_concat_all, const float* g_cross_vec,
                    float* g_x0, rk_stream_t stream);

/* Stand-alone cross_layer(x0, xl, index) (DCN/dcn.py:25-50): out = x0*(xl.w) + b + xl with
 * w, b of d floats; bwd gives g_x0 = g*(xl.w), g_xl = g + w*(g.x0). */
int rk_cross_layer_fwd(const float* x0, const float* xl, const float* w, const float* b, int d,
                       int64_t B, float* out, rk_stream_t stream);
int rk_cross_layer_bwd(const float* x0, const float* xl, const float* w, int d, int64_t B,
                       const float* g_out, float* g_x0, float* g_xl, rk_stream_t stream);

/* ---- DIN (DIN.forward DIN/din.py:294-323, din_attention :42-84) ----------------------------
 * One launch does every gather, the local activation unit on the history positions t < len,
 * the masked raw / scaled-softmax pooling, the concat and the per-sample L2 norm.
 *   concat_all[B,width] = [dense | cat rows | target row q | attention output]
 *   norm[B]   = || concat_all[b, l2_from:] ||_2      (l2_reg = lambda * mean(norm), DIN/din.py:322)
 *   att_w[B,T] = the attention weights w_t (raw masked scores or softmax), saved for backward
 *   relu_masks[B,T,3] = sign bits of the two hidden layers (64 + 32) for positions t < len
 * mlp: the per-call weights of att_net (DIN/din.py:61-67) packed as rk_din_mlp_floats(D) floats:
 *   [W1^T 4D x 64][b1 64][W2^T 64 x 32][b2 32][w3 32][b3 1, pad 3][W1 64 x 4D][W2 32 x 64]. */
typedef struct rk_din_args {
    const rk_field_t*   cat;          /* category fields; out_off = column in concat_all */
    int32_t             n_cat;
    int32_t             n_dense;
    const float* const* dense_cols;   /* host array of n_dense device pointers; value (b,c) at
                                         dense_cols[c][b * dense_stride] (the reference passes a
                                         dict of [B] tensors, DIN/din.py:296) */
    int64_t             dense_stride;
    rk_field_t          target;       /* feedid table, idx [B]; out_off = column of q */
    rk_field_t          history;      /* his_read_comment_7d_seq table, idx [B,T] */
    const int64_t*      hist_len;     /* [B] */
    int32_t             T;
    int32_t             att_off;      /* column of the attention output */
    int32_t             width;        /* row width of concat_all */
    int32_t             l2_from;      /* first column under the L2 norm */
    int32_t             use_softmax;
    int32_t             precision;    /* RK_DIN_FP32: fp32 SIMT MLP (1e-5 parity);
                                         RK_DIN_BF16_TENSOR: the activation-unit MLP on tcgen05 with
                                         bf16 operands / fp32 TMEM accumulators (D = 16, 2e-2 bar) */
    const float*        mlp;
    int64_t             B;
    void*               mlp_tiles;    /* RK_DIN_BF16_TENSOR only, required there: rk_din_tile_bytes() bytes of
                                         scratch (128-byte aligned) that rk_din_fwd fills with the split-bf16
                                         operand tiles of `mlp` for both directions (one small prologue launch);
                                         every CTA then fetches its weights with one bulk (TMA) copy.
                                         rk_din_bwd reads what the forward wrote: pass the same buffer,
                                         untouched in between. */
} rk_din_args_t;
#define RK_DIN_FP32 0
#define RK_DIN_BF16_TENSOR 1
int rk_din_tile_bytes(void);

int rk_din_mlp_floats(int D);
/* History width T: any T >= 0 with RK_DIN_FP32.  Its CTAs walk their samples' live positions in tiles of
 * at most 128 rows: samples of at most 128 positions whole, several to a tile, and a longer sample in chunks
 * (raw pooling and the softmax's running max / sum carried across chunks in a fixed order: deterministic, no
 * atomics, no host synchronisation).
 * T = 0 (every history empty) gives an attention output of 0 and needs no att_w / relu_masks / history
 * pointers.  RK_DIN_BF16_TENSOR takes 0 <= T <= 128 and refuses wider histories: use RK_DIN_FP32 there. */
int rk_din_fwd(const rk_din_args_t* args, float* concat_all, float* norm, float* att_w,
               uint32_t* relu_masks, int32_t* err_flag, rk_stream_t stream);
/* g_row[B,width]: per-occurrence gradients of every concat column (tower gradient g_concat + L2
 * term through g_norm[B] + the attention's d/dq on the target columns); g_hist[B,T,D]: per-
 * occurrence gradients of the history rows, written only where the position is live (t < len,
 * or every t of a len == 0 sample in softmax mode). */
int rk_din_bwd(const rk_din_args_t* args, const float* concat_all, const float* norm,
               const float* att_w, const uint32_t* relu_masks, const float* g_concat,
               const float* g_norm, float* g_row, float* g_hist, int32_t* err_flag,
               rk_stream_t stream);

/* ---- AFM pairwise-interaction attention pooling (AFM/afm.py:92-115, attention net :84-88) ---
 * fields: F tables of equal dim D (4..32, multiple of 4), 2 <= F <= 16; w1 [A,D], b1 [A],
 * w2 [A] (attention.2.weight is [1,A]), b2 [1]; A <= 128.  out[B,D] = sum_p softmax_p(s) v_p.
 * bwd: g_rows[B,F*D] per-occurrence embedding gradients; the gradients of the four registered
 * attention tensors are written to ONE contiguous buffer g_w1|g_b1|g_w2|g_b2; partials is scratch
 * of n_ctas * (A*D + 2A + 1) floats with n_ctas = rk_afm_bwd_ctas(B, F). */
int rk_afm_bwd_ctas(int64_t B, int F);
int rk_afm_fwd(const rk_field_t* fields, int F, const float* w1, const float* b1, const float* w2,
               const float* b2, int A, int64_t B, float* out, int32_t* err_flag, rk_stream_t stream);
int rk_afm_bwd(const rk_field_t* fields, int F, const float* w1, const float* b1, const float* w2,
               const float* b2, int A, int64_t B, const float* g_out, float* g_rows, float* g_w1,
               float* g_b1, float* g_w2, float* g_b2, float* partials, int n_ctas,
               int32_t* err_flag, rk_stream_t stream);
/* The same forward with the attention MLP on the tensor cores (tcgen05.mma, split-bf16 operands
 * hi.hi + lo.hi + hi.lo, fp32 accumulation in TMEM); same arguments and outputs as rk_afm_fwd, plus
 * `tiles` (required): rk_afm_tile_bytes() bytes of scratch (128-byte aligned) that the forward fills
 * once (one small prologue launch) with the weights' operand tiles for BOTH directions; every CTA
 * then fetches them by bulk (TMA) copy.  rk_afm_tc_bwd reads what the forward wrote: pass the
 * same buffer, untouched in between. */
int rk_afm_tile_bytes(void);
int rk_afm_tc_fwd(const rk_field_t* fields, int F, const float* w1, const float* b1, const float* w2,
                  const float* b2, int A, int64_t B, float* out, void* tiles, int32_t* err_flag,
                  rk_stream_t stream);
/* The backward on the tensor cores: same arguments and outputs as rk_afm_bwd, with
 * n_ctas = rk_afm_tc_bwd_ctas(B, F).  The hidden layer only enters through its 0/1 ReLU mask
 * (exact in bf16), the other operands are split-bf16; the weight-gradient accumulator lives in
 * TMEM for the life of a CTA and the per-CTA partials are added in a fixed order.  A ReLU
 * decision whose pre-activation lies inside the error band of the split product is recomputed
 * in fp32, so the masks are the fp32 kernel's masks and the results meet the fp32 parity bar
 * (1e-5); these two entry points are what the AFM module uses by default. */
int rk_afm_tc_bwd_ctas(int64_t B, int F);
int rk_afm_tc_bwd(const rk_field_t* fields, int F, const float* w1, const float* b1, const float* w2,
                  const float* b2, int A, int64_t B, const float* g_out, float* g_rows, float* g_w1,
                  float* g_b1, float* g_w2, float* g_b2, float* partials, int n_ctas,
                  const void* tiles, int32_t* err_flag, rk_stream_t stream);

/* ---- fused tower layers (SURVEY 8(f) item 3): Dice (DIN/din.py:26-36) and the BatchNorm1d that
 *      follows it in the DIN tower (DIN/din.py:272-285), training mode ------------------------
 * x, z: [B, units] row-major.  xh = batchnorm(x; eps1, no affine), p = sigmoid(xh),
 * y = alpha*(1-p)*x + p*x, z = gamma * batchnorm(y; eps2) + beta; gamma = beta = NULL: z = y.
 * Running statistics (may be NULL) are updated in place as nn.BatchNorm1d does (momentum,
 * unbiased variance, num_batches += 1).  stats[4, units] = mean1 | rstd1 | mean2 | rstd2 is kept
 * for the backward.  1 <= B <= rk_dice_bn_max_batch() (a CTA holds the whole batch of its
 * columns in registers; every batch statistic is a fixed-order block reduction). */
int rk_dice_bn_max_batch(void);
int rk_dice_bn_fwd(const float* x, int64_t B, int units, const float* alpha, float eps1,
                   const float* gamma, const float* beta, float eps2, float momentum1,
                   float* running_mean1, float* running_var1, int64_t* num_batches1,
                   float momentum2, float* running_mean2, float* running_var2,
                   int64_t* num_batches2, float* z, float* stats, rk_stream_t stream);
/* g_x[B, units]; g_alpha, g_gamma, g_beta: [units] (complete sums over the batch). */
int rk_dice_bn_bwd(const float* x, const float* g_z, int64_t B, int units, const float* alpha,
                   const float* gamma, const float* stats, float* g_x, float* g_alpha,
                   float* g_gamma, float* g_beta, rk_stream_t stream);

/* BatchNorm1d (affine, training mode) fused with the ReLU / LeakyReLU that follows it in the DeepFM
 * and BST towers (DeepFM/deepfm.py:100-110, BST/bst.py:203-214): z = act(gamma * batchnorm(x) + beta),
 * act(u) = u > 0 ? u : slope * u (slope 0 = ReLU, 0.01 = the BST tower, 1 = batch norm alone).
 * stats[2, units] = mean | rstd.  Same batch limit and determinism as rk_dice_bn_fwd. */
int rk_bn_act_fwd(const float* x, int64_t B, int units, const float* gamma, const float* beta,
                  float eps, float momentum, float* running_mean, float* running_var,
                  int64_t* num_batches, float slope, float* z, float* stats, rk_stream_t stream);
int rk_bn_act_bwd(const float* x, const float* g_z, int64_t B, int units, const float* gamma,
                  const float* beta, float slope, const float* stats, float* g_x, float* g_gamma,
                  float* g_beta, rk_stream_t stream);

/* Weight and bias gradients of a tower nn.Linear (y = x W^T + b): dW[N, K] = G^T X and db[N] = sum_b G[b, :],
 * on the tensor core (tcgen05) in 3xTF32 (about 22 bits of every operand, fp32 accumulation), or in fp32 FMA
 * where the batch is too small to fill half the GPU with tensor-core tiles; db is summed in double.  Row b of x[B, K] starts at x + b*ldx, of g[B, N] at g + b*ldg (ldx >= K, ldg >= N); db may be
 * NULL (no bias).  The batch is split into slabs whose partial sums a second launch adds in a fixed order:
 * partials holds rk_linear_wgrad_scratch_floats(B, K, N) floats (0: may be NULL).  Bit-identical from run to
 * run; no allocation, no synchronisation. */
int64_t rk_linear_wgrad_scratch_floats(int64_t B, int K, int N);   /* -1 for B, K or N < 1 */
int rk_linear_wgrad(const float* x, int64_t ldx, const float* g, int64_t ldg, int64_t B, int K, int N,
                    float* dW, float* db, float* partials, rk_stream_t stream);

/* ---- row-wise Adam on the touched rows of a table (SURVEY 8(f) item 3; opt-in: the reference
 *      uses dense optim.Adam, e.g. DeepFM/deepfm.py:226) ---------------------------------------
 * rows[n]: distinct row numbers, grads[n, D]: their summed gradient rows (a coalesced sparse
 * gradient: RowShardedEmbedding, nn.Embedding(sparse=True)).  torch.optim.SparseAdam's update:
 *   m += (g - m)(1 - beta1); v += (g*g - v)(1 - beta2);
 *   w -= lr * sqrt(1 - beta2^step) / (1 - beta1^step) * m / (sqrt(v) + eps)
 * on those rows of weight / exp_avg / exp_avg_sq ([V, D] each) only; step >= 1 is the global step. */
int rk_rowwise_adam(float* weight, float* exp_avg, float* exp_avg_sq, const int64_t* rows,
                    const float* grads, int64_t n, int D, int64_t V, float lr, float beta1,
                    float beta2, float eps, int64_t step, int32_t* err_flag, rk_stream_t stream);
/* The same update for a touched-rows gradient whose live count is on the device (no host sync
 * between the backward and the optimizer): rows[capacity], grads[capacity, D], only the first
 * *count (<= capacity) entries are applied.  This is what the replicated tables' opt-in sparse
 * gradients feed (rk_plan_compact_fields + rk_embgrad_segment_reduce on the rank keys). */
int rk_rowwise_adam_touched(float* weight, float* exp_avg, float* exp_avg_sq, const int64_t* rows,
                            const float* grads, const int64_t* count, int64_t capacity, int D,
                            int64_t V, float lr, float beta1, float beta2, float eps, int64_t step,
                            int32_t* err_flag, rk_stream_t stream);

/* ---- dense Adam over every parameter in one launch (the reference's optim.Adam(model.parameters(), lr),
 *      e.g. DCN/dcn.py:246), bit-identical to torch.optim.Adam(fused=True) without weight decay, amsgrad,
 *      maximize or grad scaling -------------------------------------------------------------------------
 * Per element, in fp32, with step = *step (the float32 step tensor, already incremented):
 *   m = fma(b1, m, fma(-b1, g, g));  v = fma(b2, v, fma(-b2, g*g, g*g))
 *   p -= (lr / (1 - pow(b1, step))) * m / (sqrt(v) / sqrt(1 - pow(b2, step)) + eps)
 * A tensor's gradient is either dense (grad, [rows, dim]) or a touched-rows gradient: touched_rows
 * [capacity] distinct rows in ascending order, touched_values [capacity, dim] their gradient rows, of which
 * the first *touched_count (device, clamped to [0, capacity]) are live.  Every other row takes g = 0, so its
 * moments decay as in dense Adam, with no dense gradient in memory.  Touched rows outside [0, rows) are
 * skipped and raise *err_flag (may be NULL).  param / exp_avg / exp_avg_sq / grad are contiguous fp32; lr,
 * betas and eps are per tensor, so param groups may differ within one launch.  n <= RK_ADAM_MAX_TENSORS
 * tensors per launch; no host synchronisation, capturable in a CUDA graph. */
#define RK_ADAM_MAX_TENSORS 64
typedef struct rk_adam_tensor {
    float*         param;          /* [rows, dim] */
    float*         exp_avg;
    float*         exp_avg_sq;
    const float*   step;           /* 0-d float32 */
    const float*   grad;           /* dense gradient, or NULL for a touched-rows gradient */
    const int64_t* touched_rows;
    const float*   touched_values;
    const int64_t* touched_count;  /* NULL for a dense gradient */
    int64_t        capacity;
    int64_t        rows;
    int32_t        dim;
    float          lr, beta1, beta2, eps;
    int32_t        reserved;
} rk_adam_tensor_t;
int rk_adam_step(const rk_adam_tensor_t* tensors, int n, int32_t* err_flag, rk_stream_t stream);

/* ---- row-sharded table (BASELINE config 5 "scaled": BST feedid table of 1e8 rows block-
 *      partitioned by row over the ranks; the reference itself is single-process) ------------
 * Bookkeeping around the two all-to-alls (indices out / rows back, mirrored for gradients):
 *   rk_shard_owner : owner[i] = idx[i] / rows_per_rank (out-of-range indices -> row 0 + err flag)
 *   rk_shard_route : given the stable owner-sorted order of owner[] from rk_plan_build
 *                    (sorted_owner, perm), write send_local[i] = owner-local row of the i-th sorted
 *                    request, inv[p] = sorted slot of original position p, counts[w] = requests
 *                    for rank w (W <= 64) */
int rk_shard_owner(const int64_t* idx, int64_t n, int64_t rows_total, int64_t rows_per_rank,
                   int64_t* owner, int32_t* err_flag, rk_stream_t stream);
int rk_shard_route(const int64_t* idx, const uint32_t* sorted_owner, const uint32_t* perm, int64_t n,
                   int64_t rows_total, int64_t rows_per_rank, int W, int64_t* send_local, int64_t* inv,
                   int64_t* counts, rk_stream_t stream);
/* Dense ranks of a sorted plan, for the touched-rows gradients of replicated tables (SURVEY 8(f)
 * item 3): rank_keys[i] = number of distinct rows before sorted position i, so that
 * rk_embgrad_segment_reduce run on rank_keys yields the compact [distinct rows, D] gradient.
 * sorted_keys is a whole rk_plan_build output over F fields (field f: n[f] keys, rows[f] table
 * rows).  Field f's slice of rank_keys receives keys in the layout rk_embgrad_segment_reduce
 * expects for tables of cap[f] rows (cap[f] >= the number of distinct rows; dead positions are
 * parked on cap[f]), uniq_rows its distinct rows (slice start = sum of n[g], g < f) and n_uniq[f]
 * their count.  One launch, one CTA per field, no host synchronisation. */
int rk_plan_compact_fields(const uint32_t* sorted_keys, const int64_t* n, const int64_t* rows,
                           const int64_t* cap, int F, uint32_t* rank_keys, int64_t* uniq_rows,
                           int64_t* n_uniq, rk_stream_t stream);

/* ---- DeepCrossing residual units (residual_unit + loop, DeepCrossing/deepcrossing.py:25-42,
 *      148-159), fused with the gather + concat ----------------------------------------------
 * units: n_units packed per-call weight blocks of rk_resunit_pack_floats(d, H) floats each,
 *   [W1^T d x Hp][b1 Hp][W2^T Hp x dp][b2 dp][W2 d x Hp][W1 Hp x dp], Hp = roundup(H,8),
 *   dp = roundup(d,4), zero padded (W1 [H,d], W2 [d,H] as nn.Linear stores them).
 * nets[(n_units+1), B, d]: nets[0] = the concat row, nets[i+1] = output of unit i (the last one
 * is the result; all are kept for the backward).  bwd: g_x0[B,d] = d(loss)/d(nets[0]).
 * 1 <= d, H <= 256, and the forward's block must fit the 227 KiB of shared memory a block may have
 * (e.g. d <= 151 at H = 128, d <= 88 at H = 256); the backward takes every (d, H) the forward takes. */
int rk_resunit_pack_floats(int d, int H);
int rk_resunits_fwd(const rk_field_t* fields, int F, const float* dense, int n_dense,
                    const float* units, int n_units, int H, int64_t B, float* nets,
                    int32_t* err_flag, rk_stream_t stream);
int rk_resunits_bwd(const float* nets, const float* units, int n_units, int H, int d, int64_t B,
                    const float* g_out, float* g_x0, rk_stream_t stream);

/* ---- BST transformer block (BSTTransformer.forward BST/bst.py:66-91; gather :224; pooling
 *      :238-241), d_model = 16, nhead in {1,2,4,8,16} ------------------------------------------
 * Input rows x[b,t,:] come either from a table through idx[B,T] (first block: the feedid
 * embedding) or from x_in[B,T,16] (a previous block's output).  Keys t >= seq_len[b] are masked
 * with -inf (a length-0 sample yields NaN, as in the reference).
 * Sequence length T: RK_BST_FP32 takes any T >= 1 (above 128 positions a CTA owns one sample at a time and
 * walks it in 128-row query and key chunks); RK_BST_BF16_TENSOR takes 1 <= T <= 128 and refuses a longer
 * sequence with an argument error before any CUDA call.  y_out[B,T,16] and/or the
 * pooled row sum_t y[b,t,:] (divided by seq_len[b] when pool_mean) written to
 * pool_out[b*pool_ld + 0..15] are produced.
 * Dropout (BST/bst.py:86 on w_o's output, :62 inside the FFN, :90 on the FFN output): dropout_p > 0
 * applies inverted dropout at the three sites with keep-bits that are a pure function of
 * (rng[0] = seed, rng[1] = offset, row b*T+t, site) — Philox4x32-10, 16-bit uniforms, an element is
 * dropped when its uniform < round(p*65536).  The backward regenerates the same bits from the same
 * rng values; the caller advances the offset between forwards.  The reference's own draws
 * (torch generators) cannot be replayed, so parity is defined at dropout_p = 0. */
typedef struct rk_bst_block {
    const float* pos;                                  /* position_embedding.weight [max_len,16] */
    const float *wq, *bq, *wk, *bk, *wv, *bv, *wo, *bo; /* w_q/w_k/w_v/w_o .weight [16,16], .bias [16] */
    const float *ln1_g, *ln1_b;                        /* norm1 */
    const float *w1, *b1, *w2, *b2;                    /* ffn.0, ffn.3 */
    const float *ln2_g, *ln2_b;                        /* norm2 */
    const uint64_t* rng;                               /* device [seed, offset]; may be NULL when dropout_p == 0 */
    float dropout_p;                                   /* 0 in eval mode */
    int32_t precision;                                 /* RK_BST_FP32: fp32 SIMT block (1e-5 parity); RK_BST_BF16_TENSOR: projections / FFN / weight gradients on tcgen05 (2e-2 bar) */
} rk_bst_block_t;
#define RK_BST_FP32 0
#define RK_BST_BF16_TENSOR 1

int rk_bst_grad_floats(int T);            /* T*16 + 6*256 + 10*16 */
int rk_bst_bwd_ctas(int64_t B, int T, int precision);
int rk_bst_block_fwd(const rk_bst_block_t* blk, int nhead, const float* table, const int64_t* idx,
                     int64_t table_rows, const float* x_in, const int64_t* seq_len, int64_t B, int T,
                     float* y_out, float* pool_out, int pool_ld, int pool_mean, int32_t* err_flag,
                     rk_stream_t stream);
/* g_y[B,T,16] and/or g_pool (row b at g_pool + b*g_pool_ld) -> g_x[B,T,16] and the gradients of the
 * block's registered tensors in g_params, laid out
 *   [pos T*16][wq 256][bq 16][wk][bk][wv][bv][wo][bo][ln1_g][ln1_b][w1][b1][w2][b2][ln2_g][ln2_b];
 * partials: scratch of rk_bst_bwd_ctas(B,T,blk->precision) * rk_bst_grad_floats(T) floats (for T > 128 at most
 * 2^26 floats in all). */
int rk_bst_block_bwd(const rk_bst_block_t* blk, int nhead, const float* table, const int64_t* idx,
                     int64_t table_rows, const float* x_in, const int64_t* seq_len, int64_t B, int T,
                     const float* g_y, const float* g_pool, int g_pool_ld, int pool_mean, float* g_x,
                     float* g_params, float* partials, int n_ctas, int32_t* err_flag,
                     rk_stream_t stream);

/* ---- evaluation metrics (the per-step loss.item()/label.cpu()/prob.cpu() and the per-epoch
 *      sklearn roc_auc_score / accuracy_score of train()/evaluate(), DeepFM/deepfm.py:173-180,
 *      :184-208; the challenge's per-user AUC, which the reference cannot compute) -------------
 * rk_metrics_append copies a batch of B scores / labels (fp32) and, when group != NULL, group ids
 * (int64) into score_buf / label_buf / group_buf[capacity] at offset count[0], then advances
 * count[0] (clamped to capacity).  count is int64_t[2]: count[1] is the launch's arrival counter and
 * must be 0 between launches (zero both to reset).  One launch, no host synchronisation: it may be
 * captured in a CUDA graph.  Rows past capacity are dropped.  While copying it raises bits of the
 * sticky *status: */
#define RK_METRICS_NONFINITE 1u  /* a score is NaN or infinite */
#define RK_METRICS_BAD_LABEL 2u  /* a label is not 0 or 1 */
#define RK_METRICS_BAD_GROUP 4u  /* a group id is outside [0, num_groups) */
#define RK_METRICS_OVERFLOW  8u  /* more rows than capacity were appended */
#define RK_METRICS_NOT_PROB 16u  /* a score is outside [0, 1] (log loss / accuracy are undefined) */
int rk_metrics_append(const float* score, const float* label, const int64_t* group, int64_t B,
                      float* score_buf, float* label_buf, int64_t* group_buf, int64_t capacity,
                      int64_t num_groups, int64_t* count, uint32_t* status, rk_stream_t stream);
/* rk_metrics_compute reduces the first n (< 2^31, host value) stored samples into *result (device):
 *   pos / neg   samples with label 1 / 0;  u2 = 2U, the doubled Mann-Whitney statistic with ties
 *               counted one half, so AUC = u2 / (2 pos neg) is sklearn's roc_auc_score, exactly;
 *   correct     samples with (score > 0.5) == label;  logloss_sum = sum of binary cross-entropies,
 *               each log clamped at -100 (F.binary_cross_entropy), in double, fixed order;
 *   with group != NULL (num_groups >= 1): the AUC of every group with both classes, summed in
 *   double in a fixed order (uauc_sum) over the valid_groups such groups.  Ids outside
 *   [0, num_groups), which rk_metrics_append flags, are counted as group 0.
 * Every count is an exact integer (2U <= n^2 / 2 fits uint64), so AUC does not depend on the order
 * of the samples.  ws: rk_metrics_workspace_bytes(n, num_groups) bytes (num_groups 0 without groups). */
typedef struct rk_metrics_result {
    uint64_t pos, neg, u2, correct;
    double   logloss_sum;
    uint64_t valid_groups;
    double   uauc_sum;
} rk_metrics_result_t;
size_t rk_metrics_workspace_bytes(int64_t n, int64_t num_groups);
int rk_metrics_compute(const float* score, const float* label, const int64_t* group, int64_t n,
                       int64_t num_groups, void* ws, size_t ws_bytes, rk_metrics_result_t* result,
                       rk_stream_t stream);
/* rk_metrics_merge joins the buffers of `world` data-parallel ranks, each of the same `capacity`, as an
 * all-gather lays them out: rank r's samples are score_g / label_g / group_g[r*capacity ...] and its
 * {count, arrival counter, status} are state_g[3r .. 3r+2].  Rank r's first count_r samples (count_r
 * clamped to [0, capacity], as rk_metrics_append clamps it) go to score_out / label_out / group_out at
 * offset count_0 + ... + count_{r-1}, so the storage order is rank-major; state_out gets {sum of the
 * counts, 0, OR of the statuses}, so rk_metrics_compute on the merged buffers sees every rank's samples and
 * errors.  group_g may be NULL (then group_out is not written).  Outputs must not overlap the inputs.  One
 * launch reading the counts on the device, no host synchronisation: it may be captured in a CUDA graph.
 * Refused before any CUDA call: world or capacity < 1, world*capacity >= 2^31, a NULL required pointer. */
int rk_metrics_merge(const float* score_g, const float* label_g, const int64_t* group_g, const int64_t* state_g,
                     int64_t world, int64_t capacity, float* score_out, float* label_out, int64_t* group_out,
                     int64_t* state_out, rk_stream_t stream);

/* ---- batch assembly from an encoded frame in device memory (each script's WechatDataset.__getitem__
 *      + DataLoader collation: DIN/din.py:86-222 with din_collate_fn, BST/bst.py:94-159,
 *      DCN/dcn.py:52-112, DeepFM/deepfm.py:26-70) --------------------------------------------------
 * rk_batch_gather writes one batch of B rows into caller-owned outputs.  Output row i takes source row
 * r = order[*cursor + row0 + i]: `cursor` is a device int64 the kernel reads, so a captured launch takes
 * whatever batch the cursor names when it is replayed (advance it in-stream afterwards); row0 is a
 * data-parallel rank's offset inside the global batch.
 *   cols[c]: dst row i = the row_bytes bytes of src row r (bytes are copied, never converted);
 *   seq (may be NULL): the ragged history values[offsets[r] .. offsets[r+1]) written to dst[i, 0..width)
 *            and zero-padded, its length to dst_len[i] (din_collate_fn's padding).
 * All columns are one launch; no host synchronisation.  Sticky bits of *status (no fault, and nothing is
 * written outside the outputs): */
#define RK_BATCH_MAX_COLS 32
#define RK_BATCH_WINDOW       1u  /* *cursor < 0 or *cursor + row0 + B > n_order: the batch writes nothing */
#define RK_BATCH_BAD_ROW      2u  /* an order entry is outside [0, n_rows): that row is written as zeros */
#define RK_BATCH_SEQ_OVERFLOW 4u  /* a history is longer than width: its first width ids are written and
                                     its length is written as width */
typedef struct rk_batch_col {
    const void* src;        /* [n_rows, row_bytes] */
    void*       dst;        /* [B, row_bytes] */
    int64_t     row_bytes;
} rk_batch_col_t;
typedef struct rk_batch_seq {
    const int64_t* values;  /* flat ids of every row's history */
    const int64_t* offsets; /* [n_rows + 1] */
    int64_t*       dst;     /* [B, width] */
    int64_t*       dst_len; /* [B] */
    int32_t        width;
    int32_t        reserved;
} rk_batch_seq_t;
int rk_batch_gather(const rk_batch_col_t* cols, int n_cols, const rk_batch_seq_t* seq, const int64_t* order,
                    int64_t n_order, int64_t n_rows, const int64_t* cursor, int64_t row0, int64_t B,
                    uint32_t* status, rk_stream_t stream);

/* ---- frame encoding on the device (rank_b200.loader.EncodedWechat's encode_column and DIN's history
 *      split, i.e. each script's vocabulary dict lookup per value: DIN/din.py:146-158, BST/bst.py:139-148,
 *      DCN/dcn.py:52-112, DeepFM/deepfm.py:26-70) ---------------------------------------------------------
 * A vocabulary is its n_keys unique keys (UTF-8 bytes[offsets[k] .. offsets[k+1]), each encoding to pos[k])
 * and an open-addressing table of n_slots 64-bit slots, a power of two >= 2 * n_keys (rk_vocab_slots gives
 * the smallest), which rk_vocab_build fills.  A string column is Arrow's large_string layout: row i is
 * bytes[offsets[i] .. offsets[i+1]), null when bit valid_bit0 + i of the LSB-first bitmap `valid` is 0
 * (valid may be NULL: no nulls).  Values are compared byte for byte.  Argument errors are refused before any
 * CUDA call; no entry point allocates or synchronises.  Sticky bits of *status (no fault): */
#define RK_ENCODE_TABLE_FULL  1u  /* a probe visited every slot without finding the key or an empty slot (the
                                     slots are not a table rk_vocab_build made): the key is not inserted, the
                                     value encodes to 0 */
#define RK_ENCODE_SPLIT_COUNT 2u  /* a row's item count differs from out_offsets: items past its range are
                                     not written */
typedef struct rk_vocab {
    const char*    bytes;
    const int64_t* offsets;  /* [n_keys + 1] */
    const int64_t* pos;      /* [n_keys] */
    uint64_t*      slots;    /* [n_slots] */
    int64_t        n_keys;   /* < 2^31 - 1 */
    int64_t        n_slots;
} rk_vocab_t;
typedef struct rk_str_col {
    const char*    bytes;
    const int64_t* offsets;  /* [n + 1] */
    const uint8_t* valid;    /* may be NULL */
    int64_t        valid_bit0;
    int64_t        n;
} rk_str_col_t;
/* The smallest power of two >= 2 * n_keys (at least 1); -1 for n_keys < 0 or >= 2^31 - 1. */
int64_t rk_vocab_slots(int64_t n_keys);
/* Sets every slot empty, then inserts every key (one thread per key, atomicCAS on a slot, linear probing). */
int rk_vocab_build(const rk_vocab_t* vocab, uint32_t* status, rk_stream_t stream);
/* out[i * out_stride] = pos of the key equal to row i, or 0 when there is none or the row is null
 * (encode_column).  out_stride >= 1, so a column of a wider row-major matrix is written in place. */
int rk_encode_strings(const rk_vocab_t* vocab, const rk_str_col_t* col, int64_t* out, int64_t out_stride,
                      uint32_t* status, rk_stream_t stream);
/* DIN's history split on ',' (str.split(",")), in two passes.  rk_encode_split_count: counts[i] = 1 + the
 * number of ',' bytes of row i ('' is one item, 'a,' two).  rk_encode_split: item k of row i, encoded as
 * rk_encode_strings encodes a value, to out[out_offsets[i] + k]; out_offsets is the exclusive scan of the
 * counts ([n + 1]).  Both ignore `valid` (a null history is refused by the caller, as the reference raises). */
int rk_encode_split_count(const rk_str_col_t* col, int64_t* counts, rk_stream_t stream);
int rk_encode_split(const rk_vocab_t* vocab, const rk_str_col_t* col, const int64_t* out_offsets, int64_t* out,
                    uint32_t* status, rk_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RANK_B200_H */
