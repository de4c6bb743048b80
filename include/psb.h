/*
 * psb.h -- C ABI of libpsb_b200.so: the B200 (sm_100a) implementation of the
 * embedding-scoring hot path of kepingbi/ProdSearch.
 *
 * The reference has no FFI / plugin registry: the hot path is reached through
 * PyTorch nn.Module methods (SURVEY.md 8(b)).  This header is the boundary a
 * maintainer binds instead of the ATen call sites listed per entry point
 * (paths are relative to the reference repository).  Conventions:
 *
 *   - every pointer is a DEVICE pointer unless the comment says "host";
 *   - tables and activations are row-major contiguous fp32, row length d
 *     (d % 4 == 0, d <= 512, base pointers 16-byte aligned);
 *   - indices are int64 exactly as the reference's batches carry them
 *     (data/batch_data.py:18-22); masks are uint8 (batch_data.py:174);
 *   - no entry point allocates, synchronises with the host or keeps state:
 *     work is enqueued on `stream` (a cudaStream_t) and workspace is supplied
 *     by the caller, sized by the matching *_workspace_bytes query;
 *   - return value: 0 ok, < 0 invalid argument (PSB_E_*), > 0 a cudaError_t.
 *     The Python mirror raises RuntimeError on any non-zero status, matching
 *     the reference's "plain exceptions" error behaviour (trainer.py:215).
 */
#ifndef PSB_H_
#define PSB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* psb_stream_t; /* cudaStream_t */

#define PSB_OK 0
#define PSB_E_ARG (-1)       /* null pointer / negative size */
#define PSB_E_DIM (-2)       /* d not a multiple of 4 or > 512, k out of range */
#define PSB_E_WORKSPACE (-3) /* workspace too small */
#define PSB_E_ALIGN (-4)     /* pointer not 16-byte aligned */
#define PSB_E_UNSUPPORTED (-5)

#define PSB_ABI_VERSION 1

int psb_abi_version(void);
const char* psb_status_string(int status);
/* Number of kernels this library has launched since load (host counter; lets
 * bench.py report gpu_launches without a profiler). */
int64_t psb_launch_count(void);

/* Per-kernel timing without an external profiler.  While enabled, every kernel this library launches
 * outside CUDA-graph capture is bracketed by two CUDA events on its own stream.  psb_profile_dump
 * synchronises the device, writes one text line per kernel name -- "name launches total_ms min_ms max_ms" --
 * into buf (host, NUL-terminated; returns the byte count, < 0 on error) and clears the record.
 * Host-side state: not thread-safe, meant for bench.py's roofline leg and tests. */
int psb_profile_enable(int32_t on);
int64_t psb_profile_dump(char* buf /* host */, int64_t cap);

/* ------------------------------------------------------------------ G1 ---
 * out[i,:] = table[idx[i],:]                                   (bit-exact copy)
 * Replaces aten::embedding at models/item_transformer.py:449,:464-469,:262-263,
 * :269; models/ps_model.py:257,:261,:303,:326-332; models/PV.py:53,:58;
 * models/PVC.py:76,:84.  Out-of-range indices set *err_flag (optional) to 1 and
 * produce a zero row (the reference raises IndexError on the host). */
int psb_gather_rows(const float* table, int64_t table_rows, int64_t d,
                    const int64_t* idx, int64_t n, float* out,
                    int32_t* err_flag, psb_stream_t stream);

/* ------------------------------------------------------------------ G4 ---
 * Fused gather + masked mean (+ optional dropout multiplier, + optional
 * tanh(W x + b) "fs" projection): models/text_encoder.py:6-16 get_vector_mean,
 * :75-82 AVGEncoder.forward, :32-40 FSEncoder.forward, on rows gathered by
 * models/item_transformer.py:449-450, models/ps_model.py:257-258,
 * models/PVC.py:57-60,:76-79.
 *
 *   valid[i,j] = mask ? mask[i,j] != 0 : (pad_idx < 0 || idx[i,j] != pad_idx)
 *   mean[i,:]  = sum_j valid * tok_scale[i,j] * table[idx[i,j],:] / max(#valid,1)
 *   mean      *= keep_scale[i,:]           (dropout mask already scaled by 1/(1-p))
 *   out[i,:]   = fs_weight ? tanh(fs_weight . mean[i,:] + fs_bias) : mean[i,:]
 *
 * tok_scale implements the PVC corruption (0 or 1/(1-rate), PVC.py:46-54).
 * mean_out (optional unless fs_weight given) receives the post-dropout mean
 * that the backward pass needs; inv_count (optional) receives 1/max(#valid,1). */
int psb_gather_meanpool_fwd(const float* table, int64_t table_rows, int64_t d,
                            const int64_t* idx, int64_t n, int64_t w, int64_t pad_idx,
                            const uint8_t* mask, const float* tok_scale,
                            const float* keep_scale,
                            const float* fs_weight, const float* fs_bias,
                            float* mean_out, float* out, float* inv_count,
                            psb_stream_t stream);

/* Backward of the fs projection (autograd of text_encoder.py:35-39):
 *   dz = grad_out * (1 - out^2); grad_weight[j,k] = sum_i dz[i,j] mean[i,k];
 *   grad_bias[j] = sum_i dz[i,j]; grad_mean[i,k] = keep_scale * sum_j dz[i,j] W[j,k].
 * Sums over i run in ascending i (deterministic).  The word-table gradient is a
 * scatter-reduce contribution (src = grad_mean, src_div = w, scale = valid/count). */
int psb_fs_bwd(const float* grad_out, const float* out, const float* mean,
               const float* keep_scale, const float* fs_weight, int64_t n, int64_t d,
               float* grad_weight, float* grad_bias, float* grad_mean,
               psb_stream_t stream);

/* Per-token weights valid/max(#valid,1) used by the scatter-reduce contribution of a
 * mean-pool: tok_weight[i,j] (the PVC quirk: the corruption scale is NOT applied in
 * backward, SURVEY.md 8(a) A7). */
int psb_meanpool_token_weights(const int64_t* idx, int64_t n, int64_t w, int64_t pad_idx,
                               const uint8_t* mask, float* tok_weight, psb_stream_t stream);

/* --------------------------------------------------------------- G3 / A4 ---
 * Fused gather + dot + bias + BCE-with-logits negative-sampling loss, forward and
 * the analytic score gradient in one pass.  Covers
 *   item_to_words        models/item_transformer.py:260-283  (anchor = product row)
 *   ParagraphVector      models/PV.py:57-65                   (anchor = review row)
 *   PVC                  models/PVC.py:83-91                  (anchor = corrupted mean)
 *   TEM score+loss tail  models/item_transformer.py:485,:493-514
 *                        (anchor_a = pos_out, anchor_b = neg_out, w = 1)
 *
 *   x[i,j,0]   = <anchor_a[i], table[pos_idx[i,j]]> (+ bias[pos_idx[i,j]])
 *   x[i,j,1+c] = <anchor(i,c), table[neg_idx[i,j,c]]> (+ bias[...]),
 *                anchor(i,c) = anchor_b ? anchor_b[i*k+c] : anchor_a[i]
 *   l[i,j]     = pos_weight*bce(x0,1) + sum_c nw[i,c]*bce(x_c,0)
 *   valid[i,j] = mask ? mask[i,j] : (pad_idx < 0 || pos_idx[i,j] != pad_idx)
 *   loss[i]    = sum_j valid*l[i,j] / max(#valid,1)
 *   coef_pos[i,j]   = d loss[i] / d x[i,j,0],  coef_neg[i,j,c] = d loss[i] / d x[i,j,1+c]
 *   grad_anchor_a[i,:] = sum coef * row  over the scores that used anchor_a[i]
 *   grad_anchor_b[i*k+c,:] = coef_neg[i,0,c] * table[neg_idx[i,0,c]]
 * bce(x,t) = max(x,0) - x t + log1p(exp(-|x|)); its derivative sigmoid(x) - t. */
int psb_ns_loss_fwd(const float* anchor_a, const float* anchor_b,
                    const float* table, int64_t table_rows, int64_t d, const float* bias,
                    const int64_t* pos_idx, const int64_t* neg_idx,
                    const uint8_t* mask, int64_t pad_idx,
                    const float* neg_weight, float pos_weight,
                    int64_t n, int64_t w, int64_t k,
                    float* loss, float* coef_pos, float* coef_neg,
                    float* grad_anchor_a, float* grad_anchor_b,
                    psb_stream_t stream);

/* The TEM score + loss tail (models/item_transformer.py:485,:493-514) straight from the fused encoder's output
 * block: enc_out [n, 1 + k, d] holds, per sample, the encoder output of the positive sequence and of its k negative
 * copies (psb_encoder_fwd with copies = 1 + k).  Same arithmetic as psb_ns_loss_fwd(anchor_a = enc_out[:, 0],
 * anchor_b = enc_out[:, 1:], w = 1) without the two repacking copies; coef_pos / coef_neg / grad_enc_out
 * ([n, 1 + k, d], the gradient of  grad_scale * sum_i loss_rows[i]  with respect to enc_out) come out multiplied by
 * grad_scale -- 1 / n for the reference's .mean() (:514).  k <= 7, d <= 128. */
int psb_tem_loss_fwd(const float* enc_out, const float* table, int64_t table_rows, int64_t d, const float* bias,
                     const int64_t* pos_idx /* [n] */, const int64_t* neg_idx /* [n, k] */, float pos_weight,
                     int64_t n, int64_t k, float grad_scale, float* loss_rows /* [n] */, float* coef_pos /* [n] */,
                     float* coef_neg /* [n, k] */, float* grad_enc_out, psb_stream_t stream);
/* *loss_out = mean(ps_rows[0..n_ps)) + mean(il_rows[0..n_il)) (ps_loss + item_loss, :515-520), fixed summation order;
 * *acc_ps += mean(ps_rows), *acc_il += mean(il_rows): the running sums the trainer prints (trainer.py:88-98; the
 * reference adds .item() values on the host).  acc pointers may be NULL; n_il may be 0. */
int psb_tem_loss_finish(const float* ps_rows, const float* il_rows, int64_t n_ps, int64_t n_il, float* loss_out,
                        float* acc_ps, float* acc_il, psb_stream_t stream);

/* scores[i,c] = <anchor[i], table[idx[i,c]]> (+ bias[idx[i,c]]): candidate scoring of
 * test_dotproduct (models/item_transformer.py:141-145) for an explicit candidate list
 * idx [n, c_per] (the reference's 500-candidate segments, item_pv_dataset.py:65-68). */
int psb_score_rows(const float* anchor, const float* table, int64_t table_rows, int64_t d,
                   const float* bias, const int64_t* idx, int64_t n, int64_t c_per, float* scores,
                   psb_stream_t stream);

/* ------------------------------------------------------------------ G2 ---
 * Deterministic embedding backward: sort-then-segmented-reduce instead of float
 * atomics.  Replaces aten::embedding_dense_backward (autograd of every K1 site).
 * A table's gradient is the sum of "contributions"; contribution c adds, for
 * each slot i < n:
 *     grad[idx[i], :] += s(i) * src[row(i), :]
 *     row(i) = src_row ? src_row[i] : i / src_div
 *     s(i)   = (scale ? scale[i] : 1) * (scale2 ? scale2[i / scale2_div] : 1)
 * and, when to_bias != 0, bias_grad[idx[i]] += s(i) (word_bias / product_bias,
 * item_transformer.py:272-275,:495-499).  Slots whose idx equals drop_idx (the
 * table's padding_idx: nn.Embedding zeroes that gradient row) are skipped.
 * Within one destination row the terms are added in ascending (contribution,
 * slot) order, so results are bit-reproducible and independent of the grid. */
typedef struct psb_contrib {
  const int64_t* idx;     /* [n] destination rows */
  int64_t n;
  const float* src;       /* [*, d] source rows */
  const int64_t* src_row; /* optional [n] */
  int64_t src_div;        /* used when src_row == NULL (>= 1) */
  const float* scale;     /* optional [n] */
  const float* scale2;    /* optional [ceil(n / scale2_div)] */
  int64_t scale2_div;     /* >= 1 */
  int32_t to_bias;
  int32_t reserved;
} psb_contrib_t;

#define PSB_MAX_CONTRIBS 8

int64_t psb_scatter_reduce_workspace_bytes(int64_t n_total, int64_t table_rows);

/* contribs: HOST array of n_contribs descriptors (device pointers inside).
 * Outputs: unique_rows[u] ascending, reduced[u,:], reduced_bias[u] (each optional,
 * capacity n_total), *n_unique (device int32).  If dense_grad / dense_bias_grad are
 * given, row unique_rows[u] of them is OVERWRITTEN with the reduced value (the
 * caller keeps the rest zero, see psb_zero_rows). */
int psb_scatter_reduce_rows(const psb_contrib_t* contribs, int32_t n_contribs,
                            int64_t table_rows, int64_t d, int64_t drop_idx,
                            void* workspace, int64_t workspace_bytes,
                            int32_t* unique_rows, float* reduced, float* reduced_bias,
                            int32_t* n_unique, float* dense_grad, float* dense_bias_grad,
                            psb_stream_t stream);

/* The same in two calls, so that the SORT -- which only reads the index lists -- can run long before the gradient
 * values exist (on a side stream next to the backward pass; the index tensors of a training step are all known when
 * its forward pass ends): psb_scatter_sort_rows reads only idx / n of the contributions and leaves the sorted slots,
 * segment table, unique_rows and n_unique in the workspace / outputs; psb_scatter_reduce_sorted, given contributions
 * with the SAME idx / n in the SAME order and the same workspace, runs the segmented reduce.  Together they produce
 * bit for bit what psb_scatter_reduce_rows produces.  ONE reduce per sort: the reduce consumes the workspace (its
 * list of segments that span work units is appended to, not rebuilt), so sort again before reducing again. */
int psb_scatter_sort_rows(const psb_contrib_t* contribs /* host; idx and n only */, int32_t n_contribs,
                          int64_t table_rows, int64_t drop_idx, void* workspace, int64_t workspace_bytes,
                          int32_t* unique_rows, int32_t* n_unique, psb_stream_t stream);
int psb_scatter_reduce_sorted(const psb_contrib_t* contribs /* host */, int32_t n_contribs, int64_t table_rows,
                              int64_t d, int64_t drop_idx, void* workspace, int64_t workspace_bytes,
                              const int32_t* unique_rows, float* reduced, float* reduced_bias,
                              const int32_t* n_unique, float* dense_grad, float* dense_bias_grad,
                              psb_stream_t stream);

/* dense[rows[u], :] = 0 (and dense_bias[rows[u]] = 0) for u < *n_rows: clears the
 * rows a previous step touched so a persistent dense .grad costs O(batch). */
int psb_zero_rows(const int32_t* rows, const int32_t* n_rows, int64_t max_rows,
                  int64_t d, float* dense, float* dense_bias, psb_stream_t stream);

/* ------------------------------------------------------------------ G5 ---
 * Full-catalog scoring with fused top-k: S = Q . E^T (+ bias), top-k per query,
 * ties broken by LOWER item id.  Replaces test_dotproduct
 * (models/item_transformer.py:111-146) + Trainer.get_prod_scores
 * (trainer.py:189-226) + host argsort (trainer.py:136,:152) for the TEM path; the
 * [M, N] score matrix is never materialised.
 *   queries [m, d], table [n_items, d] (rows >= n_items, e.g. the pad row, are not
 *   candidates), bias optional [n_items], id_base/id_stride map local row r to
 *   the global item id id_base + r * id_stride (row-sharded catalogs).
 * Outputs: out_ids [m, k] int64 (-1 where fewer than k candidates), out_scores
 * [m, k] fp32, descending score / ascending id.
 * mode: PSB_TOPK_EXACT  fp32 FFMA scoring (reference arithmetic, CUDA cores)
 *       PSB_TOPK_TC     tcgen05 TF32 shortlist + exact fp32 rescoring (same result) */
#define PSB_TOPK_EXACT 0
#define PSB_TOPK_TC 1
#define PSB_TOPK_TC16 2 /* workspace query only: psb_catalog_topk_f16 takes the prepared fp16 copy */

int64_t psb_catalog_topk_workspace_bytes(int64_t m, int64_t n_items, int64_t d, int64_t k, int32_t mode);
int psb_catalog_topk(const float* queries, int64_t m, const float* table, int64_t n_items,
                     int64_t d, const float* bias, int64_t k, int64_t id_base, int64_t id_stride,
                     int32_t mode, const float* max_row_sqnorm, void* workspace, int64_t workspace_bytes,
                     int64_t* out_ids, float* out_scores, psb_stream_t stream);

/* max_r |table[r,:]|^2 as a device scalar: the bound the TC mode's error margin needs.  Pass it
 * to psb_catalog_topk (max_row_sqnorm) to skip the extra table pass when the table is static
 * (evaluation); NULL there makes the call compute it itself. */
int psb_table_max_row_sqnorm(const float* table, int64_t rows, int64_t d, float* out,
                             psb_stream_t stream);

/* fp16 shortlist on a half-precision COPY of a static (evaluation) table -- same results as the exact mode.
 * psb_catalog_prepare_f16 converts table[0..n_items) to fp16 (round to nearest) into table_f16 [n_items, d] and
 * writes stats[0] = max_r |e_r|^2, stats[1] = max_r |e_r - half(e_r)|^2, stats[2] = 1 if a value does not fit
 * fp16 (stats: 4 device floats, 16-byte aligned).  psb_catalog_topk_f16 then shortlists with tcgen05 kind::f16
 * (half the table bytes per pass, up to 512 queries per pass over the table), bounds the shortlist error from the
 * MEASURED quantisation errors, and rescoring the survivors exactly in fp32 from `table` as PSB_TOPK_TC does.
 * A table that overflows fp16 (stats[2] != 0) makes every row take the exact streaming fallback: still correct,
 * slow -- callers use PSB_TOPK_TC for such tables.  Workspace: psb_catalog_topk_workspace_bytes(mode TC16). */
int psb_catalog_prepare_f16(const float* table, int64_t n_items, int64_t d, void* table_f16, float* stats,
                            psb_stream_t stream);
int psb_catalog_topk_f16(const float* queries, int64_t m, const float* table, const void* table_f16,
                         const float* stats, int64_t n_items, int64_t d, const float* bias, int64_t k,
                         int64_t id_base, int64_t id_stride, void* workspace, int64_t workspace_bytes,
                         int64_t* out_ids, float* out_scores, psb_stream_t stream);

/* Debug aid: TMEM read rate of tcgen05.ld.32x32b.x32 issued back to back by `warps` (1..16) warps of one CTA,
 * in bytes per SM clock -- bytes_per_clk[0] with one CTA on the GPU, [1] with one CTA per SM.  The catalog
 * contraction (K = 128) reads every accumulator element back after 8 MMAs, so this rate bounds its tensor-pipe
 * utilisation.  Synchronises the device, allocates and frees 20 KB.  bytes_per_clk: 2 doubles (host). */
int psb_debug_tmem_read_bw(int32_t warps, int32_t iters, double* bytes_per_clk);

/* Debug aid: out[m, j] = a[m, k] . bt[j, k]^T (+ bias[j]) on tcgen05 with the 3xTF32 split (csrc/gemm3_tf32.cu) --
 * the tensor-core form of the encoder's linear layers (models/neural.py:118-120 linear_keys / linear_values /
 * linear_query; models/transformer.py:37-88), which the FFMA kernels compute on the FFMA path (PSB_ENC_TC=0).
 * k % 64 == 0, j % 64 == 0, lda % 4 == 0, ldo % 4 == 0, 16-byte aligned pointers; PSB_E_UNSUPPORTED otherwise.  The
 * encoder uses it for the q and K|V projections and the backward's grad-xn product on the tensor-core path (the
 * default). */
int psb_debug_gemm3_tf32(const float* a, int64_t lda, int64_t m, int64_t k, const float* bt, int64_t j,
                         const float* bias, float* out, int64_t ldo, psb_stream_t stream);
/* Debug aid: with PSB_FT_TRACE=1 in the environment the fused tensor-core encoder tail (tail_fused_tc_kernel,
 * csrc/gemm3_tf32.cu) and its backward counterpart (tail_bwd_fused_tc_kernel) stamp %globaltimer (ns) at their phase
 * boundaries in CTA 0; this copies the 64 stamps of the last launches (forward 0..31, backward 32..63) to the host
 * (synchronising).  PSB_E_UNSUPPORTED when tracing is off. */
int psb_debug_tail_trace(uint64_t* out64 /* host */);

/* Merge g per-shard top-k lists (ids [g, m, k], scores [g, m, k], as all_gather
 * lays them out) into the global top-k with the same ordering rule. */
int psb_topk_merge(const int64_t* ids, const float* scores, int64_t g, int64_t m, int64_t k,
                   int64_t* out_ids, float* out_scores, psb_stream_t stream);

/* ------------------------------------------------------------------ N1 ---
 * Fused single-layer sequence encoder restricted to ONE output position: the last
 * TransformerEncoderLayer + final LayerNorm of models/transformer.py:37-88 as used by
 * ItemTransformerRanker.forward_dotproduct / test_dotproduct
 * (models/item_transformer.py:478-491,:118-140) and ProductRanker (models/ps_model.py:336-339),
 * which read only top_vecs[:, out_pos, :].  Per input sequence s (S of them, T tokens):
 *
 *   x[t]   = valid[t] * in[t] + pe[t]                      (transformer.py:75-80)
 *   xn[t]  = pre_ln ? LayerNorm_attn(x[t]) : x[t]          (transformer.py:47-50; layer 0: no LN)
 *   K,V    = xn Wk^T + bk, xn Wv^T + bv; q = (xn[o] Wq^T + bq) / sqrt(d/heads)   (neural.py:190-205)
 *   P[h,:] = softmax_t(q_h . K_h[t], masked -> -1e18)      (neural.py:206-213)
 * and per copy c < copies (the reference re-encodes the SAME sequence for the positive and
 * every negative item, item_transformer.py:478-487; only the dropout masks differ):
 *   ctx    = sum_t drop1(P)[h,t] V_h[t];  y = drop2(ctx Wo^T + bo) + x[o]         (neural.py:222-226, transformer.py:56)
 *   z      = drop4(drop3(gelu(LN_ff(y) W1^T + b1)) W2^T + b2) + y                 (neural.py:30-33)
 *   out[s*copies + c, :] = LayerNorm_out(z)                                        (transformer.py:86)
 * Tokens: either first[s] (token 0) followed by table[idx[s, t-1]] (valid iff idx != pad_idx)
 * -- the TEM layout [query, purchased items] -- or a dense [S,T,d] tensor with a uint8 mask
 * (1 = real token; NULL = all real).  Masked keys get probability exactly 0; a sequence with no
 * valid token attends uniformly, as the reference's softmax over equal -1e18 scores does.
 * Dropout uses Philox4x32-10 keyed by *seed_dev (device uint64; a CUDA-graph replay sees the new
 * seed), stream 1..4 = {attention, context, ff inner, ff output}, element index as laid out
 * above; p_drop == 0 disables it.  All arithmetic fp32 (FFMA), fixed summation order.
 * Shapes supported: d % 4 == 0, d <= 128, ff % 4 == 0, ff <= 1024, T <= 64, d % heads == 0, heads <= 32,
 * copies <= 24.  The backward tail keeps the attention scores of a tile of R >= copies rows (R in {16, 20, 24}) in
 * shared memory, which bounds heads * T; past it the calls return PSB_E_UNSUPPORTED.  At d = 128, ff = 512 the
 * bound is heads * T <= 847 for copies <= 16, <= 511 for copies <= 20 and <= 282 for copies <= 24 (8 heads: any
 * T <= 64 up to 20 copies, T <= 35 at 21..24 copies). */
typedef struct psb_encoder_params {
  /* nn.Linear layout [out, in]; names follow models/neural.py / models/transformer.py */
  const float *wq, *bq, *wk, *bk, *wv, *bv, *wo, *bo;
  const float *ln_attn_g, *ln_attn_b; /* TransformerEncoderLayer.layer_norm (pre_ln only) */
  const float *ln_ff_g, *ln_ff_b;     /* feed_forward.layer_norm */
  const float *w1, *b1, *w2, *b2;     /* feed_forward.w_1 [ff,d], w_2 [d,ff] */
  const float *ln_out_g, *ln_out_b;   /* TransformerEncoder.layer_norm */
} psb_encoder_params_t;

typedef struct psb_encoder_grads { /* same shapes; every pointer is OVERWRITTEN (not accumulated) */
  float *wq, *bq, *wk, *bk, *wv, *bv, *wo, *bo;
  float *ln_attn_g, *ln_attn_b, *ln_ff_g, *ln_ff_b, *w1, *b1, *w2, *b2, *ln_out_g, *ln_out_b;
} psb_encoder_grads_t;

typedef struct psb_encoder_cfg {
  int64_t S, T, d, heads, ff, copies, out_pos; /* out_pos in [0, T) */
  int32_t pre_ln;
  int32_t raw_input; /* dense input only: rows are a previous layer's output -- the mask removes KEYS but
                        rows are not zeroed and pe is not added (layers > 0 of a deeper encoder) */
  float ln_eps, p_drop;
  const uint64_t* seed_dev; /* device; required when p_drop > 0 */
  const float* first;       /* [S,d] token 0, with table/idx [S,T-1] for tokens 1.. */
  const float* table;
  int64_t table_rows;
  const int64_t* idx;
  int64_t pad_idx;
  const float* dense;       /* alternative input [S,T,d] (first/table/idx NULL) */
  const uint8_t* mask;      /* [S,T] for the dense input */
  const float* pe;          /* [T,d] positional rows or NULL (use_pos False) */
  void* first_ready;        /* optional cudaEvent_t (forward only): `first` is being produced on ANOTHER stream and
                               this event marks its completion; the call enqueues its token plan and weight
                               transposes (which do not read `first`) and makes `stream` wait for the event only
                               before the first kernel that does -- the query pooling overlaps with them */
  void* wgrad_done;         /* optional cudaEvent_t (backward only): the WEIGHT gradients (split-M partial products +
                               their fixed-order reduce: nothing on the data-gradient path needs them) are computed on
                               a library-owned side stream, forked after the tail kernel, and this event is recorded
                               behind them.  grad_first / grad_rest / grad_dense are complete in `stream` order as
                               usual; the CALLER makes every consumer of `grads` (and the release of `workspace`) wait
                               for the event.  NULL: everything runs on `stream`. */
} psb_encoder_cfg_t;

/* Byte sizes of the caller-owned buffers: `saved` carries forward state to the backward call,
 * `workspace` is scratch (backward != 0: size for psb_encoder_bwd).  < 0: invalid cfg. */
int64_t psb_encoder_saved_bytes(const psb_encoder_cfg_t* cfg);
int64_t psb_encoder_workspace_bytes(const psb_encoder_cfg_t* cfg, int32_t backward);

/* out [S*copies, d].  cfg / params are HOST structs holding device pointers. */
int psb_encoder_fwd(const psb_encoder_cfg_t* cfg, const psb_encoder_params_t* params,
                    void* saved, int64_t saved_bytes, void* workspace, int64_t workspace_bytes,
                    float* out, psb_stream_t stream);

/* Backward of psb_encoder_fwd for grad_out [S*copies, d] (same cfg, params, saved buffer).
 * grad_first [S,d] + grad_rest [S,T-1,d] (TEM layout; rows of invalid tokens are zero) or
 * grad_dense [S,T,d]; parameter gradients into `grads` (NULL members are skipped). */
int psb_encoder_bwd(const psb_encoder_cfg_t* cfg, const psb_encoder_params_t* params,
                    const void* saved, int64_t saved_bytes, void* workspace, int64_t workspace_bytes,
                    const float* grad_out, float* grad_first, float* grad_rest, float* grad_dense,
                    const psb_encoder_grads_t* grads, psb_stream_t stream);

/* ------------------------------------------------------------------ N2 ---
 * Fused global-norm clip + Adam over all parameter tensors of the model: replaces
 * clip_grad_norm_(params, max_grad_norm) + torch.optim.Adam(eps=1e-9).step() as driven by
 * models/optimizers.py:205-243 (noam schedule :214-219 when noam != 0).  Dense semantics, identical
 * to the reference: every element of every tensor is updated every step.
 *   total = sqrt(sum_t |g_t|^2); c = min(1, max_grad_norm / (total + 1e-6))   (max_grad_norm <= 0: c = 1)
 *   g' = c g (+ weight_decay p); m += (1-b1)(g' - m); v = b2 v + (1-b2) g'^2
 *   p -= lr_t / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps),  t = ++(*step_dev)
 * No host sync: t, total^2 (sqnorm_dev, readable afterwards) live in device memory, so the call
 * replays inside a CUDA graph.  Gradients are NOT rescaled in place.  Hyper-parameters are doubles, as the
 * reference passes them: 1 - beta and the bias corrections are formed in double and then rounded, like torch. */
typedef struct psb_adam_tensor {
  float* p;
  const float* g;
  float* m;
  float* v;
  int64_t n;
} psb_adam_tensor_t;

#define PSB_ADAM_MAX_TENSORS 64

int64_t psb_adam_workspace_bytes(const psb_adam_tensor_t* tensors /* host */, int32_t n_tensors);
int psb_adam_step(const psb_adam_tensor_t* tensors /* host */, int32_t n_tensors, double lr, double beta1,
                  double beta2, double eps, double weight_decay, double max_grad_norm, int32_t noam,
                  double warmup_steps, int32_t norm_given, int64_t* step_dev, float* sqnorm_dev, void* workspace,
                  int64_t workspace_bytes, psb_stream_t stream);
/* norm_given != 0: *sqnorm_dev already holds the GLOBAL squared gradient norm (row-sharded training: the
 * caller sums psb_grad_sqnorm of every rank's shard gradients and of the replicated ones) and is used as is;
 * norm_given == 2: *step_dev has been advanced by the caller as well (psb_peer_sum_sqnorm). */

/* *sqnorm_out (device) = sum over the tensors' gradients of |g|^2, fixed summation order.  Workspace as for
 * psb_adam_step. */
int psb_grad_sqnorm(const psb_adam_tensor_t* tensors /* host; only g and n are read */, int32_t n_tensors,
                    float* sqnorm_out, void* workspace, int64_t workspace_bytes, psb_stream_t stream);

/* Row-sparse Adam for embedding tables (SURVEY.md 8(f) N2 as written: "consume G2's (unique_rows, grad_rows)
 * directly ... lazy per-row step counters").  Replaces, for the tables, the dense sweep of
 * torch.optim.Adam(eps=1e-9) + clip_grad_norm_ (models/optimizers.py:186,:205-243) by work proportional to the rows
 * a step touches, with DENSE-EQUIVALENT results: a row that rests for k steps is brought up to date when it is next read or
 * updated -- with a zero gradient its moments decay geometrically, so the skipped updates are a series with
 * independent terms: the first min(k, psb_adam_catchup_steps) are summed with each step's own coefficients (they
 * shrink like (b1/sqrt(b2))^j and are below 1e-9 of the first one after that), the moments decay in closed form by
 * the factors a dense step applies, (1 - fl(1-b1))^k and fl(b2)^k.  A step in which a table has no row list (it is
 * not passed, or has no valid entry) is a zero-gradient step for all of its rows, as in a dense step with a zero
 * gradient.  last_step == 0 means "never updated, moments zero": a caller that restores moments from a checkpoint
 * taken at step t stamps every row with t.  weight_decay is not supported here (use psb_adam_step).  The global clip
 * norm is taken over the dense tensors' gradients plus the compact row gradients (all other rows have gradient zero). */
typedef struct psb_adam_rows {
  float* p;                /* [table_rows, d] the table                                                      */
  float* m;                /* [table_rows, d] exp_avg                                                        */
  float* v;                /* [table_rows, d] exp_avg_sq                                                     */
  int32_t* last_step;      /* [table_rows] optimizer step up to which the row (and its bias element) is current */
  const int32_t* rows;     /* [cap] unique rows with a gradient this step (psb_scatter_reduce_rows unique_rows) */
  const float* grad;       /* [cap, d] their reduced gradients                                               */
  const int32_t* n_rows;   /* device scalar: valid entries of rows / grad / bias_grad                        */
  int64_t cap, d, table_rows;
  float* bias_p;           /* optional [table_rows] bias vector indexed like the table (product_bias, word_bias) */
  float* bias_m;
  float* bias_v;
  const float* bias_grad;  /* [cap] or NULL (bias present but without gradient this step)                    */
  int32_t grad_by_row;     /* 0: grad / bias_grad are compact lists (entry i belongs to rows[i]); 1: they are DENSE
                            * [table_rows, d] / [table_rows] buffers of which only the listed rows are valid (the
                            * owner-side fold of a row-sharded table writes such a buffer)                        */
  int32_t reserved;
} psb_adam_rows_t;

#define PSB_ADAM_MAX_ROW_TABLES 8
#define PSB_ADAM_MAX_IDX_LISTS 8

/* Terms of the catch-up series summed per resting row for these betas (198 at 0.9 / 0.999). */
int32_t psb_adam_catchup_steps(double beta1, double beta2);
int64_t psb_adam_sparse_workspace_bytes(const psb_adam_tensor_t* dense /* host */, int32_t n_dense,
                                        const psb_adam_rows_t* tables /* host */, int32_t n_tables);
/* One optimizer step: dense tensors exactly as psb_adam_step, tables through their row lists.  coef_hist: device
 * array of coef_cap float2 (8-byte aligned) the call appends this step's (lr_t / (1 - b1^t), 1 / sqrt(1 - b2^t)) to
 * -- also when n_tables == 0 -- and reads earlier steps' values from (steps >= coef_cap are recomputed on the fly);
 * may be NULL.  Every step of a run that catches rows up through coef_hist must pass it.  norm_given as in
 * psb_adam_step. */
int psb_adam_sparse_step(const psb_adam_tensor_t* dense /* host */, int32_t n_dense,
                         const psb_adam_rows_t* tables /* host */, int32_t n_tables, double lr, double beta1,
                         double beta2, double eps, double max_grad_norm, int32_t noam, double warmup_steps,
                         int32_t norm_given, int64_t* step_dev, float* sqnorm_dev, float* coef_hist, int64_t coef_cap,
                         void* workspace, int64_t workspace_bytes, psb_stream_t stream);
/* |g|^2 over the dense tensors' gradients plus the row lists of the tables (the first phase of psb_adam_sparse_step on
 * its own: row-sharded training publishes this partial norm to the peers).  Workspace as for psb_adam_sparse_step. */
int psb_grad_sqnorm_sparse(const psb_adam_tensor_t* dense /* host; g and n */, int32_t n_dense,
                           const psb_adam_rows_t* tables /* host */, int32_t n_tables, float* sqnorm_out,
                           void* workspace, int64_t workspace_bytes, psb_stream_t stream);
/* Bring rows up to the current step (*step_dev) BEFORE they are read: idx_lists[0..n_lists) are device index arrays
 * (the ones the forward pass is about to gather with), idx_counts their lengths (host); n_lists == 0 catches up every
 * row of the table (before evaluation / a checkpoint).  skip_row: a row that never moves (the pad row) or -1.
 * Only p / m / v / last_step / bias_* / d / table_rows of ``table`` are read. */
int psb_adam_rows_catchup(const psb_adam_rows_t* table /* host */, const int64_t* const* idx_lists /* host array */,
                          const int64_t* idx_counts /* host */, int32_t n_lists, int64_t skip_row, double lr,
                          double beta1, double beta2, double eps, int32_t noam, double warmup_steps,
                          const int64_t* step_dev, const float* coef_hist, int64_t coef_cap, psb_stream_t stream);

/* ------------------------------------------------------------ multi-GPU ---
 * Row-sharded tables over NVLink peer memory (SURVEY.md 8(e)): owner of row id = id % G, local row =
 * id / G.  One process per GPU; buffers that peers read (table shards, gradient staging lists, the flat
 * dense-gradient bucket, barrier flags) are allocated with psb_peer_alloc, exported as a 64-byte handle that
 * the host side exchanges (torch.distributed all_gather), and opened by every other rank: after that a peer
 * buffer is an ordinary device pointer and the exchange is plain loads inside the kernels below.  Replaces
 * the index / row / gradient all-to-alls of the NCCL transport (prodsearch_b200/sharded.py).  No entry point
 * synchronises with the host, so a whole multi-GPU training step replays as one CUDA graph per rank. */
#define PSB_PEER_HANDLE_BYTES 64
#define PSB_PEER_MAX 16

int psb_peer_alloc(int64_t bytes, void** out /* host */);      /* cudaMalloc + zero fill (IPC-exportable) */
int psb_peer_free(void* p);
int psb_peer_export(void* p, void* handle /* host, 64 bytes */);
int psb_peer_open(const void* handle /* host */, void** out /* host */); /* maps the peer allocation, enables P2P */
int psb_peer_close(void* p);

/* Cross-GPU barrier on the launching streams of all G ranks.  flag_blocks: HOST array of G device pointers,
 * flag_blocks[r] = rank r's flag block (uint32[PSB_PEER_MAX], zero-initialised peer memory).  *epoch_dev (local
 * device uint32, starts at 0) counts the barriers of this rank.  A rank that waits longer than timeout_cycles
 * (<= 0: about 2 s) stops waiting and writes 1 + the missing peer into *err_dev instead of hanging.
 * wait_cycles_dev (optional, uint64[4]): SM cycles this rank spent inside the barrier are added to
 * wait_cycles_dev[wait_slot & 3] -- how long a rank waits for its peers at each barrier of a replayed step. */
int psb_peer_barrier(const void* const* flag_blocks, int32_t rank, int32_t G, uint32_t* epoch_dev,
                     int32_t* err_dev, int64_t timeout_cycles, uint64_t* wait_cycles_dev, int32_t wait_slot,
                     psb_stream_t stream);

/* out[i,:] = shard[idx[i] % G][idx[i] / G, :]: the forward "fetch" of a row-sharded table (bit-exact copies,
 * 128-bit loads over NVLink for remote owners) into a local mini table.  shards: HOST array of G device
 * pointers.  remap_out (optional, [n]): the position each index is read at afterwards, remap_out[i] =
 * idx[i] == pad_id ? pad_pos : i, so that all pad entries share ONE mini-table position and the consuming
 * kernels keep their "idx != pad_idx" validity rule; the rows of pad entries other than position pad_pos are
 * then not fetched (out is zero there). */
int psb_peer_gather_rows(const void* const* shards, int32_t G, int64_t rows_total, int64_t d,
                         const int64_t* idx, int64_t n, float* out, int64_t* remap_out, int64_t pad_id,
                         int64_t pad_pos, int32_t* err_flag, psb_stream_t stream);

/* Owner-side gradient fold.  Every rank r publishes a compact list in peer memory -- the unique_rows / reduced /
 * n_unique outputs of its psb_scatter_reduce_rows over GLOBAL row ids.  For every row this rank owns
 * (id % G == rank, local row id / G) that occurs in at least one list:
 *     dense[id / G, :] = scale * sum_r vals_r[slot_r(id), :]      (r ascending: reproducible, no atomics)
 * in two launches for up to two tables, independent of G: "mark" writes (stamp, slot) of every owned slot into
 * posmap[r][local]; "sum" lets the lowest peer holding a row add the later peers' rows and OVERWRITE the dense
 * row once.  Rows no list holds are not written: the caller keeps them zero (psb_zero_rows with the `touched`
 * list of the previous fold, or a memset).  *stamp_dev must be constant during the call and differ from the
 * previous call's value (the barrier epoch); posmap is uint64[G * shard_rows], zero-initialised once. */
typedef struct psb_fold_table {
  const int32_t* rows[PSB_PEER_MAX];   /* per peer: [cap] ascending unique global ids (peer memory) */
  const float* vals[PSB_PEER_MAX];     /* per peer: [cap, d] */
  const int32_t* n_rows[PSB_PEER_MAX]; /* per peer: device count */
  int64_t cap, d, shard_rows;
  void* posmap;
  float* dense;                        /* [shard_rows, d] */
  int32_t* touched;                    /* optional [G * cap]: local rows written, unordered */
  int32_t* n_touched;                  /* device counter for `touched` (caller zeroes it) */
} psb_fold_table_t;

/* psb_peer_gather_rows for a table whose owners update it with the row-sparse Adam: a row that rests on its owner
 * (last_step < *step_dev) is brought up to date ON THE FLY by the reader -- it loads the row's moments as well and adds
 * the catch-up series (psb_adam_rows_catchup's arithmetic) to the value it hands out -- WITHOUT writing anything back:
 * the owner's copy is only ever written by the owner's own optimizer step (which catches the row up first), so no
 * cross-GPU write, no lock.  shards_p / _m / _v / _last: G peer pointers each ([local_rows, d] fp32 x3, [local_rows]
 * int32); step_dev / coef_hist: this rank's step counter and coefficient history (identical on every rank). */
int psb_peer_gather_rows_lazy(const void* const* shards_p, const void* const* shards_m, const void* const* shards_v,
                              const void* const* shards_last, int32_t G, int64_t rows_total, int64_t d,
                              const int64_t* idx, int64_t n, float* out, int64_t* remap_out, int64_t pad_id,
                              int64_t pad_pos, int32_t* err_flag, double lr, double beta1, double beta2, double eps,
                              int32_t noam, double warmup_steps, const int64_t* step_dev, const float* coef_hist,
                              int64_t coef_cap, psb_stream_t stream);
int psb_peer_fold_lists(const psb_fold_table_t* tables /* host */, int32_t n_tables, int32_t rank, int32_t G,
                        float scale, const uint32_t* stamp_dev, psb_stream_t stream);

/* out[i] = scale * sum_r bufs[r][i], added in ascending r (one-shot all-reduce of the replicated dense
 * gradients; every rank computes the identical sum) but LOADED starting at the caller's own rank, so the G
 * readers never all pull from the same GPU at once.  bufs: HOST array of G device pointers (peer memory). */
int psb_peer_allreduce(const void* const* bufs, int32_t G, int32_t rank, int64_t n, float scale, float* out,
                       psb_stream_t stream);

/* *sqnorm_out = sum_r *slots[r] (r ascending): the GLOBAL squared gradient norm from the partial norms every rank
 * published (psb_grad_sqnorm of its shard gradients; rank 0 adds the replicated ones).  step_dev != NULL: the
 * optimizer's step counter is advanced here, for psb_adam_step(norm_given = 2). */
int psb_peer_sum_sqnorm(const void* const* slots, int32_t G, float* sqnorm_out, int64_t* step_dev,
                        psb_stream_t stream);

/* psb_grad_sqnorm(_sparse) + psb_peer_barrier + psb_peer_sum_sqnorm as ONE chain with a single tail launch: the partial
 * sums of this rank's gradients (dense tensors and row lists, as psb_grad_sqnorm_sparse), then one kernel that finishes
 * them, publishes the shard norm in slots[rank], runs the cross-GPU barrier, adds the G slots in rank order into
 * *sqnorm_out and advances *step_dev (for psb_adam_step / psb_adam_sparse_step with norm_given = 2).  Barrier arguments
 * as psb_peer_barrier; workspace as psb_adam_sparse_workspace_bytes. */
int psb_peer_norm_exchange(const psb_adam_tensor_t* dense /* host; g and n */, int32_t n_dense,
                           const psb_adam_rows_t* tables /* host */, int32_t n_tables, const void* const* slots,
                           const void* const* flag_blocks, int32_t rank, int32_t G, uint32_t* epoch_dev,
                           int32_t* err_dev, int64_t timeout_cycles, uint64_t* wait_cycles_dev, int32_t wait_slot,
                           float* sqnorm_out, int64_t* step_dev, void* workspace, int64_t workspace_bytes,
                           psb_stream_t stream);

/* ------------------------------------------------------------------ N4 ---
 * On-device batch construction, metrics ranks and the ranklist writer for the item-transformer (TEM) path
 * (SURVEY.md 8(f) N4).  The corpus relations the reference keeps as nested Python lists
 * (data/data_util.py:165-203) live in HBM as flat CSR arrays; one launch replaces the per-sample list
 * comprehensions of ItemPVDataloader.get_train_batch / get_test_batch / get_user_review_idxs
 * (data/item_pv_dataloader.py:122-143,:31-49,:85-105). */
typedef struct psb_corpus {
  const int32_t* review_user;    /* [n_reviews] review -> user   (global_data.review_u_p[r][0]) */
  const int32_t* review_item;    /* [n_reviews] review -> item   (global_data.review_u_p[r][1]) */
  const int32_t* review_uloc;    /* [n_reviews] position in the user's sequence (review_loc_time[r][0]); may be
                                    NULL unless mode == PSB_HIST_SEQ */
  const uint8_t* review_in_set;  /* [n_reviews] 1 = review of the training split (prod_data.u_reviews) */
  const int64_t* user_seq_off;   /* [n_users + 1] CSR offsets into user_seq */
  const int32_t* user_seq;       /* every user's reviews in time order (global_data.u_r_seq) */
  const int64_t* item_query_off; /* [n_items + 1] CSR offsets into item_query (prod_data.product_query_idx) */
  const int32_t* item_query;
  const int64_t* query_words;    /* [n_queries, wq] padded with word_pad (global_data.query_words) */
  int64_t n_reviews, n_users, n_items, n_queries, wq, word_pad;
  /* review-transformer (RTM) batches only; NULL otherwise */
  const int64_t* item_seq_off;   /* [n_items + 1] CSR offsets into item_seq */
  const int32_t* item_seq;       /* every item's reviews in time order (global_data.i_r_seq) */
  const int64_t* review_time;    /* [n_reviews] time stamp (review_loc_time[r][2]); PSB_HIST_SEQ only */
} psb_corpus_t;

#define PSB_HIST_SEQ 0    /* do_seq_review_*: the hist_limit reviews before this one (item_pv_dataloader.py:88-91) */
#define PSB_HIST_LAST 1   /* fix=True: last hist_limit training reviews of the user, this one excluded (:93-97) */
#define PSB_HIST_RANDOM 2 /* fix=False: random subset of hist_limit, order kept (:98-101); the subset is the
                             hist_limit candidates with the smallest psb_subset_key(seed, sample, position) */

/* corpus: HOST struct of device pointers.  Per sample b: review_idx[b] (the purchase being predicted);
 * user_idx / item_idx [batch] optional (NULL: taken from the review, as get_train_batch does; test batches
 * supply them, item_pv_dataset.py:66); query_idx [batch] optional -- when NULL the query is
 * item_query[item][query_pick[b] % n] (random.choice at item_pv_dataloader.py:131 with the random word
 * supplied by the caller).  Outputs: target_prod_idxs [batch], query_idx_out [batch] (optional),
 * query_word_idxs [batch, wq], u_item_idxs [batch, hist_limit] right-padded with item_pad (the reference pads
 * to the batch maximum, util.pad: slice [:, :max(hist_len)] to reproduce its width), hist_len [batch].
 * Samples with out-of-range ids come out all-pad and set *err_flag (optional). */
int psb_build_item_batch(const psb_corpus_t* corpus /* host */, const int64_t* review_idx,
                         const int64_t* user_idx, const int64_t* item_idx, const int64_t* query_idx,
                         const uint32_t* query_pick, int64_t batch, int64_t hist_limit, int32_t mode,
                         uint32_t seed, int64_t item_pad, int64_t* target_prod_idxs, int64_t* query_idx_out,
                         int64_t* query_word_idxs, int64_t* u_item_idxs, int32_t* hist_len, int32_t* err_flag,
                         psb_stream_t stream);

/* N3: candidate sequences of a review-transformer TEST batch (ProdSearchDataLoader.get_test_batch,
 * data/prod_search_dataloader.py:44-109, which loops over every candidate of every entry in Python).  One warp per
 * (entry b, candidate c): the user's previous reviews (get_user_review_idxs, :184-201; PSB_HIST_LAST or
 * PSB_HIST_SEQ, at most u_limit) followed by the candidate item's reviews (get_item_review_idxs, :135-160, fix=True,
 * at most i_limit; PSB_HIST_SEQ: those not later than the entry review's time stamp, dataset.bisect_right).
 * width = u_limit + i_limit.  Outputs, laid out [batch, n_cand, ...]:
 *   ridxs [.., width]      review ids, right-padded with review_pad
 *   seg   [.., width + 1]  0 (query slot), 1 per user review, 2 per item review, then seg_pad
 *   users [.., width + 1]  user_pad, the entry's user per user review, each item review's author, then user_pad
 *   items [.., width + 1]  item_pad, each user review's item, the candidate per item review, then item_pad
 *   seq_len [batch, n_cand] number of reviews (optional)
 * A candidate id < 0 (the reference's -1 padding of short candidate lists, :92) yields an all-pad row (seg all
 * seg_pad), exactly what util.pad_3d(dim=1) appends.  The reference pads to the batch maximum: slice
 * [..., :max(seq_len)] (+1) to reproduce its width. */
int psb_build_review_test_batch(const psb_corpus_t* corpus /* host */, const int64_t* review_idx,
                                const int64_t* user_idx, const int64_t* candi_prod_idxs, int64_t batch,
                                int64_t n_cand, int64_t u_limit, int64_t i_limit, int32_t mode,
                                int64_t review_pad, int64_t user_pad, int64_t item_pad, int64_t seg_pad,
                                int64_t* ridxs, int64_t* seg, int64_t* users, int64_t* items, int32_t* seq_len,
                                int32_t* err_flag, psb_stream_t stream);

/* The subset key of PSB_HIST_RANDOM, evaluated on the host (tests, oracle cross-check). */
uint32_t psb_subset_key(uint32_t seed, uint32_t sample, uint32_t pos);

/* rank[i] = 1-based position of target[i] in ids[i, :k], 0 if absent: the input of MRR / P@1
 * (Trainer.calc_metrics, trainer.py:171-186) taken from the fused top-k lists. */
int psb_target_rank(const int64_t* ids, const int64_t* target, int64_t m, int64_t k, int32_t* rank,
                    psb_stream_t stream);

/* TREC run file of Trainer.test (trainer.py:158-169): for every query i and rank r < min(cutoff, k)
 * "%s_%d Q0 %s %d %f ReviewTransformer\n" % (user_ids[user_idx[i]], query_idx[i], product_ids[ids[i,r]],
 * r + 1, scores[i,r]).  ALL pointers are HOST pointers (ids / scores: the [m, k] top-k lists copied back).
 * A negative id ends a query's list.  Returns the number of lines written (< 0: PSB_E_*). */
int64_t psb_write_ranklist(const char* path, const char* const* user_ids, const int64_t* user_idx,
                           const int64_t* query_idx, const char* const* product_ids, const int64_t* ids,
                           const float* scores, int64_t m, int64_t k, int64_t cutoff, int32_t append);

#ifdef __cplusplus
}
#endif
#endif /* PSB_H_ */
