/*
 * llamarec_b200 -- C ABI of the B200-native (sm_100a) implementation of LlamaRec's stage-1
 * candidate-generation hot path and the stage-2 verbalizer tail.
 *
 * The reference (GarciaLnk/LlamaRec) is pure Python/PyTorch and has NO plugin/FFI boundary; the
 * reference interface each entry point replaces is the Python call site cited beside it
 * (paths relative to the reference tree).  INTEGRATION.md shows the ctypes binding a maintainer
 * of the reference would add.
 *
 * Conventions
 *   - every function returns int: 0 = OK, >0 = cudaError_t, <0 = lrb error (LRB_ERR_*);
 *     lrb_last_error() returns a thread-local human-readable message for the last failure.
 *   - all data pointers are caller-owned DEVICE pointers, contiguous, 16-byte aligned, unless the
 *     parameter name ends in _host.  Nothing is allocated internally; scratch is passed in and its
 *     size comes from the matching *_workspace_bytes / *_slots query.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *     asynchronous with respect to the host and safe to capture in a CUDA graph.
 *   - no global mutable state; re-entrant across streams and devices.
 *   - the hidden width is fixed at d = 64 (LRURec default `bert_hidden_units`, config.py:212).
 */
#ifndef LLAMAREC_B200_H_
#define LLAMAREC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRB_OK 0
#define LRB_ERR_BAD_ARG (-1)
#define LRB_ERR_UNSUPPORTED (-2)
#define LRB_ERR_WORKSPACE (-3)
#define LRB_ERR_DRIVER (-4)
#define LRB_ERR_ARCH (-5)

#define LRB_D 64          /* embedding width                                        */
#define LRB_H 128         /* complex LRU state width (2*d), model/lru.py:105         */
#define LRB_FF 256        /* PFFN inner width (4*d), model/lru.py:96                 */
#define LRB_MAX_LEN 256   /* max sequence length (ML-100k uses 200, config.py:59)    */
#define LRB_MAX_K 50      /* max top-k list length (= max of metric_ks, config.py:137) */

const char* lrb_last_error(void);
int lrb_version(void);

/* Queries the device the calling thread is bound to: number of SMs and compute capability
 * (major*10+minor).  Kernels refuse to launch (LRB_ERR_ARCH) on anything but sm_100. */
int lrb_device_info(int* num_sms, int* cc);

/* ------------------------------------------------------------------------------------------
 * Item table preparation (once per model load / per shard).
 * Replaces nothing at run time; it lays out `embedding.token.weight` (model/lru.py:50) and
 * `model.bias` (model/lru.py:71) for the scoring kernels:
 *   table_bf16 [rows][64]  bf16 copy of table_f32 rows [row_begin, row_begin+rows)
 *   bias_pad   [ceil(rows/256)*256] fp32 copy of bias, -inf in the padding
 *   bias_blk   (optional, may be NULL) ceil(rows/256)*8192 bytes: the bias folded into a K=16 bf16
 *              slab (hi/mid/lo split) that the tensor-core kernel multiplies by a block of ones,
 *              so its epilogue never adds a bias.  Pass NULL to lrb_score_topk when the bias is
 *              identically zero (the reference's initial state, model/lru.py:71).
 * ------------------------------------------------------------------------------------------ */
size_t lrb_bias_blk_bytes(int64_t rows);
int lrb_prepare_table(const float* table_f32, const float* bias_f32, int64_t row_begin,
                      int64_t rows, void* table_bf16, float* bias_pad, void* bias_blk, void* stream);

/* ------------------------------------------------------------------------------------------
 * Sequence preparation: one pass over the id matrix.
 * Replaces LRUEmbedding.get_mask (model/lru.py:54-55), the power-of-two left pad
 * (model/lru.py:75-78) and the history mask of trainer/lru.py:36-38 (as a sorted exclusion list).
 *   ids        [B][L] int64 (the reference's LongTensors) or int32 (pre-padded device eval sets),
 *              id_bytes = 8 or 4; 0 = padding (dataloader/lru.py:147-149 left-pads)
 *   all_positions = 0: eval mode, tokens before the first non-zero id are skipped
 *                 = 1: every position is a token (forward() at all L positions)
 * Outputs
 *   tok_first  [B]  first position that is a token
 *   tok_offset [B+1] exclusive prefix sum of token counts (tok_offset[B] = total tokens)
 *   excl_sorted [B][excl_stride] ascending ids to exclude (history + id 0), INT32_MAX padded;
 *               excl_stride = lrb_excl_stride(L).  May be NULL (no exclusion list wanted).
 *   excl_bloom [B][4] 128-bit filter over (id & 127).  NULL iff excl_sorted is NULL.
 * ------------------------------------------------------------------------------------------ */
int lrb_excl_stride(int L);
int lrb_prepare_sequences(const void* ids, int id_bytes, int B, int L, int all_positions,
                          int32_t* tok_first, int32_t* tok_offset, int32_t* excl_sorted,
                          uint32_t* excl_bloom, void* stream);

/* ------------------------------------------------------------------------------------------
 * LRURec encoder.  Replaces LRUEmbedding.forward + LRUModel.forward up to (not including) the
 * scoring matmul: model/lru.py:57-60, 73-83, 149-161, 173-175.
 *
 * `weights` is the packed fp32 parameter blob described by lrb_encoder_weight_floats() /
 * llamarec_b200/packing.py (embedding LayerNorm, then per block: lambda re/im, gamma, W_in^T,
 * b_in, W_out^T (real part form), b_out, LN, W1^T, b1, W2^T, b2, LN).
 *   ids / id_bytes: the id matrix handed to lrb_prepare_sequences (int64 or int32, consumed as is)
 *   table_f32 [N+1][64] fp32 embedding table (gathered by id)
 *   all_positions = 0: u[B][64] = hidden state at the last position (eval / retrieval)
 *                 = 1: hidden[B][L][64] at every position (train-step forward)
 *   out_bf16 (optional, eval mode only): bf16 copy of u, [B][64], feeds lrb_score_topk
 * Workspace: lrb_encode_workspace_bytes(B, L, all_positions).
 * ------------------------------------------------------------------------------------------ */
size_t lrb_encoder_weight_floats(int n_blocks);
size_t lrb_encode_workspace_bytes(int B, int L, int all_positions);
int lrb_encode_fwd(const void* ids, int id_bytes, int B, int L, const float* table_f32, int64_t table_rows,
                   const float* weights, int n_blocks, int all_positions,
                   const int32_t* tok_first, const int32_t* tok_offset, float* out_f32,
                   void* out_bf16, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Catalogue scoring fused with a streaming per-user top-K.
 * Replaces `x @ E^T + bias` (model/lru.py:85) at the last position, the history mask
 * (trainer/lru.py:36-38) and torch.topk (trainer/lru.py:82-84, demo/inference.py:49).
 *
 * The kernel emits `slots` partial lists per user (one per item-range split); lrb_merge_metrics
 * reduces them (and, after an all-gather, the lists of other ranks) to the final top-K.
 *   precision 0 (bf16): u_bf16 [B][64] bf16, table_bf16 [rows][64] bf16 -- tcgen05 tensor cores
 *   precision 1 (fp32): u_f32  [B][64] fp32, table_f32  [rows][64] fp32 -- exact FFMA path for
 *                       small catalogues (bit-comparable with the fp32 reference).  While a block of
 *                       >= 128 users' score rows fits in the scratch buffer (rows <= ~560 k) the scores are
 *                       written out once and one warp per user applies the history mask and selects the
 *                       top K with a radix select -- literally scores[b, history] = -inf; torch.topk
 *                       (trainer/lru.py:36-38,82-84) -- and ONE sorted list per user comes out (slots == 1);
 *                       beyond that a streaming kernel emits one partial list per item-range split
 *   bias_pad / bias_blk: from lrb_prepare_table (fp32 path reads bias_pad; bf16 path reads bias_blk,
 *   NULL = zero bias).  row_offset: global id of local row 0 (row sharding).
 *   excl_sorted/excl_bloom/excl_stride: from lrb_prepare_sequences, NULL = no exclusion
 *   (BaseTrainer.validate calls calculate_metrics(exclude_history=False), trainer/base.py:141).
 * Outputs (caller allocated): part_scores/part_ids [B][slots][K], part_cnt [B][slots];
 *   scratch: lrb_score_scratch_bytes(B) (both precisions).
 * ------------------------------------------------------------------------------------------ */
int lrb_score_topk_slots(int B, int64_t rows, int precision, int* slots);
size_t lrb_score_scratch_bytes(int B);
int lrb_score_topk(const void* u, const void* table, const float* bias_pad, const void* bias_blk,
                   int B, int64_t rows, int64_t row_offset, const int32_t* excl_sorted, const uint32_t* excl_bloom,
                   int excl_stride, int K, int precision, float* part_scores, int32_t* part_ids,
                   int32_t* part_cnt, int slots, void* scratch, void* stream);

/* Dense scores for API-compatible LRURec.forward (model/lru.py:85): out[M][ld_out] fp32,
 * out[m][n] = x[m,:] . table[n,:] + bias[n] for n < rows.  precision as above (1 = exact fp32). */
int lrb_score_dense(const void* x, const void* table, const float* bias_pad, const void* bias_blk,
                    int64_t M, int64_t rows, int precision, float* out, int64_t ld_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Train-step forward loss without the logits tensor.
 * Replaces, in value, LRUTrainer.calculate_loss (trainer/lru.py:22-28): `model(seqs).view(-1, N+1)`
 * followed by nn.CrossEntropyLoss(ignore_index=0) (trainer/lru.py:20) -- an online log-sum-exp over
 * the catalogue fused with the scoring contraction (exact fp32 path).
 *   hidden [M][64] fp32: encoder output at every position (lrb_encode_fwd, all_positions = 1), M = B*L
 *   table_f32 [rows][64], bias_pad: as for lrb_score_dense (rows = N+1, the whole table)
 *   labels [M] int64; rows whose label == ignore_index do not count.  Neither does a row whose label
 *   is outside [0, rows): this call does not synchronise, so it cannot raise the error torch's
 *   cross_entropy raises for such a label (lrb_train_step does); the row only leaves the mean.
 * Outputs: row_loss [M] (optional, 0 for rows that do not count); loss_sum[2] += {sum of row losses,
 *   counted rows} (the caller zeroes it; mean loss = loss_sum[0] / loss_sum[1]).
 * Workspace: lrb_ce_workspace_bytes(M, rows).
 * ------------------------------------------------------------------------------------------ */
size_t lrb_ce_workspace_bytes(int64_t M, int64_t rows);
int lrb_ce_loss_fwd(const float* hidden, const float* table_f32, const float* bias_pad, int64_t M, int64_t rows,
                    const int64_t* labels, int64_t ignore_index, float* row_loss, float* loss_sum,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Train step: loss AND the gradient of every parameter, without the logits tensor.
 * Replaces LRUTrainer.calculate_loss + loss.backward() (trainer/lru.py:22-28, trainer/base.py:107-111),
 * i.e. the backward of model/lru.py:38-41,57-60,73-86,149-161,173-175 under
 * nn.CrossEntropyLoss(ignore_index) (trainer/lru.py:20), in eval mode: no dropout (lrb_train_step_dropout
 * below is the train-mode step; this function is that call with every rate 0).  Rows must be
 * left-padded (dataloader/lru.py:98-118) -- otherwise LRB_ERR_UNSUPPORTED.
 *   ids [B][L] int64/int32 (id_bytes 8/4), labels [B*L] int64: each is ignore_index or in [0, table_rows),
 *   like the targets torch's cross_entropy accepts -- otherwise LRB_ERR_BAD_ARG (found on the device: the
 *   outputs are then meaningless)
 *   table_f32 [table_rows][64], bias_f32 [table_rows], weights = the packed blob of lrb_encode_fwd,
 *   params_log [n_blocks][3][128] (nu_log, theta_log, gamma_log of every block, model/lru.py:119)
 * Outputs (overwritten)
 *   loss_sum [2]      sum of the row losses, number of counted rows (loss = [0] / [1])
 *   grad_weights      lrb_encoder_weight_floats(n_blocks) floats, laid out like `weights`; the
 *                     lambda_re / lambda_im / gamma slots hold d nu_log / d theta_log / d gamma_log
 *   grad_table [table_rows][64]  (scoring matmul + embedding gather: the table is tied)
 *   grad_bias  [table_rows]
 * Workspace: lrb_train_workspace_bytes(B, L, n_blocks).  Synchronises the stream once (the error flag of the
 * two input checks above).
 * ------------------------------------------------------------------------------------------ */
size_t lrb_train_workspace_bytes(int B, int L, int n_blocks);
int lrb_train_step(const void* ids, int id_bytes, const int64_t* labels, int B, int L, const float* table_f32,
                   int64_t table_rows, const float* bias_f32, const float* weights, const float* params_log,
                   int n_blocks, int64_t ignore_index, float* loss_sum, float* grad_weights, float* grad_table,
                   float* grad_bias, void* workspace, size_t workspace_bytes, void* stream);

/* Train step with the reference's train-mode dropout (model/lru.py:47-52,93-97 build the modules):
 *   site 0        embedding dropout on the gathered row, before the LayerNorm (:57-60)     width 64,  p_embed
 *   site 1 + 3i   block i, dropout(out_proj(h).real) before the residual add (:160)      width 64,  p_attn
 *   site 2 + 3i   block i, dropout(gelu(w_1(x))) (:174)                                   width 256, p_ffn
 *   site 3 + 3i   block i, dropout(w_2(x_)) before the residual add (:175)               width 64,  p_ffn
 * (p_embed = p_ffn = bert_dropout, p_attn = bert_attn_dropout in the reference.)  The masks are counter-based:
 * element (t, j) of site s, t = b*L + l, is kept iff word (j & 3) of
 *   Philox4x32-10(counter = (t, j >> 2, s, 0), key = (seed & 0xffffffff, seed >> 32))   (Random123 constants)
 * is >= floor(double(p) * 2^32), and a kept element is scaled by 1.0f / (1.0f - p).  The backward recomputes the
 * masks; nothing is stored, and the workspace is lrb_train_workspace_bytes(B, L, n_blocks).  A rate of 0 turns its
 * site off exactly.  Every rate must satisfy 0 <= p < 1 (NaN too is rejected): LRB_ERR_BAD_ARG otherwise.
 * torch's own dropout RNG stream is not reproduced; lrb_dropout_mask gives the masks. */
int lrb_train_step_dropout(const void* ids, int id_bytes, const int64_t* labels, int B, int L, const float* table_f32,
                           int64_t table_rows, const float* bias_f32, const float* weights, const float* params_log,
                           int n_blocks, int64_t ignore_index, float* loss_sum, float* grad_weights,
                           float* grad_table, float* grad_bias, void* workspace, size_t workspace_bytes,
                           void* stream, float p_embed, float p_attn, float p_ffn, uint64_t seed);

/* Keep bits of one dropout site of lrb_train_step_dropout: keep[t][j] (device, T x width bytes) = 1 if element
 * (t, j) survives, 0 if it is dropped -- the same device function the train-step kernels evaluate.  Lets a caller
 * reproduce a step outside the library.  0 <= p < 1, T >= 1, width >= 1, site >= 0. */
int lrb_dropout_mask(uint64_t seed, int site, int T, int width, float p, uint8_t* keep, void* stream);

/* ------------------------------------------------------------------------------------------
 * k-way merge + Recall/MRR/NDCG + candidate emission, one fused kernel.
 * Replaces absolute_recall_mrr_ndcg_for_ks (trainer/utils.py:43-90), the label membership test and
 * candidate list of LRUTrainer.generate_candidates (trainer/lru.py:82-88, 114-132).
 *   lists: `n_lists` sorted lists per user, list j of user b at  scores[(j*list_stride_j + b*list_stride_b) ...]
 *          i.e. element i = base + j*stride_list + b*stride_user + i ; cnt likewise without i
 *          (cnt may be NULL = every list holds K_in entries).  This covers both the
 *          [B][slots][K] layout of lrb_score_topk and the [R][B][K] layout after an all-gather.
 *   labels [B] int64 (NULL = no metrics)     ks [n_ks] host array, ascending or not
 * Outputs
 *   top_scores/top_ids [B][K_out]  sorted by (score desc, id asc); missing entries = (-inf, -1);
 *                consecutive users are out_stride elements apart (0 = K_out, i.e. dense), so both
 *                arrays can live interleaved in one exchange payload [B][2][K_out]
 *   label_rank [B] int32: 0-based rank of the label in the merged list, -1 if absent
 *   metric_sums [3*n_ks] fp32: per k (in the order given) sum over users of Recall, MRR, NDCG
 *                (accumulated: the caller zeroes it once per epoch / per batch as it prefers)
 * ------------------------------------------------------------------------------------------ */
int lrb_merge_metrics(const float* list_scores, const int32_t* list_ids, const int32_t* list_cnt,
                      int n_lists, int64_t stride_list, int64_t stride_user, int64_t cnt_stride_list,
                      int64_t cnt_stride_user, int K_in, int B, int K_out, const int64_t* labels,
                      const int32_t* ks_host, int n_ks, float* top_scores, int32_t* top_ids,
                      int64_t out_stride, int32_t* label_rank, float* metric_sums, void* stream);

/* ------------------------------------------------------------------------------------------
 * Peer-memory exchange of the row-sharded, data-parallel retrieval step (one process per GPU; the
 * buffers are mapped into every process of the node over NVLink/NVSwitch).  The reference has no
 * multi-device retrieval path (SURVEY section 2.1, 8e); these replace the all-gather of user states
 * and the all-to-all of local top-K lists a collective library would run around lrb_score_topk.
 *
 * lrb_peer_push: "all-gather by stores".  Copies n_arrays local arrays (bytes_host[a] bytes each, a
 *   multiple of 16) to n_dst destinations each: dst_host[a*n_dst + d] is where array a lands on
 *   destination d (this rank's slot of peer d's gather buffer; may be local or peer-mapped memory).
 * lrb_merge_metrics_scatter: lrb_merge_metrics whose output rows are scattered by owner: user b's
 *   merged list goes to row (b % users_per_dst) of destination b / users_per_dst
 *   (dst_scores_host[d] / dst_ids_host[d], rows out_stride elements apart) -- the all-to-all fused
 *   into the merge that produces its payload.  No labels / metrics in this variant.
 * Ordering between ranks (a barrier after the stores, double-buffered destinations) is the caller's.
 * ------------------------------------------------------------------------------------------ */
int lrb_peer_push(const void* const* src_host, const size_t* bytes_host, int n_arrays,
                  void* const* dst_host, int n_dst, void* stream);
int lrb_merge_metrics_scatter(const float* list_scores, const int32_t* list_ids, const int32_t* list_cnt,
                              int n_lists, int64_t stride_list, int64_t stride_user, int64_t cnt_stride_list,
                              int64_t cnt_stride_user, int K_in, int B, int K_out,
                              float* const* dst_scores_host, int32_t* const* dst_ids_host, int n_dst,
                              int users_per_dst, int64_t out_stride, void* stream);

/* ------------------------------------------------------------------------------------------
 * Stage-2 verbalizer tail.  Replaces lm_head on the last position (model/llm.py:113-114,131) and
 * ManualVerbalizer.process_logits (trainer/verb.py:546-586: project -> [normalize -> log] ->
 * aggregate) by computing only the label-word rows of the lm_head.
 *   hidden  [B][H] bf16 last-position hidden states     lm_head [V][H] bf16
 *   word_ids [C][W] int32 first sub-token id of each label word, word_mask [C][W] (0/1)
 *   mode 0 = raw label logits (post_log_softmax=False, the reference default, trainer/llm.py:96)
 *        1 = log(softmax over all C*W label words + 1e-15)   (post_log_softmax=True)
 *   round_bf16 != 0: round each logit to bf16 first, as a bf16 lm_head GEMM followed by
 *                    .float() does (model/llm.py:113-114)
 *   calib_logits: NULL, or [V] fp32 = ManualVerbalizer._calibrate_logits (register_calibrate_logits,
 *                 trainer/verb.py:202-208): in mode 1 the label-word probabilities are divided by the
 *                 calibration vector's own label-word probabilities (+1e-15) and renormalised over all
 *                 label words before the log (ManualVerbalizer.calibrate, trainer/verb.py:616-643)
 *   out [B][C] fp32 : masked mean over the W words of each class (trainer/verb.py:611-614)
 * ------------------------------------------------------------------------------------------ */
int lrb_verbalizer_score(const void* hidden_bf16, const void* lm_head_bf16, int B, int H, int64_t V,
                         const int32_t* word_ids, const uint8_t* word_mask, int C, int W, int mode,
                         int round_bf16, const float* calib_logits, float* out, void* stream);

/* ManualVerbalizer.process_logits on logits that already exist (trainer/verb.py:546-586, the call of
 * trainer/llm.py:68 and demo/inference.py:68): logits [B][ld] fp32 (ld >= V), tok_ids/tok_mask
 * [C][W][T] (sub-tokens of every label word), word_mask [C][W]; handler = handle_multi_token
 * (trainer/verb.py:280-305): 0 first, 1 max, 2 mean; mode and calib_logits as above (the calibration vector goes
 * through the same handler).  out [B][C]. */
int lrb_verbalizer_from_logits(const float* logits, int64_t ld, int B, int64_t V, const int32_t* tok_ids,
                               const uint8_t* tok_mask, const uint8_t* word_mask, int C, int W, int T,
                               int handler, int mode, const float* calib_logits, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LLAMAREC_B200_H_ */
