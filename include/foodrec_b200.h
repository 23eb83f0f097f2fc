/*
 * foodrec_b200 -- C ABI of the B200-native graph-propagation + full-ranking hot path.
 *
 * The reference (sdu-zyx/Multi-modal-Food-Recommendation, "FoodRec/...") is pure Python and has no
 * FFI of its own; each entry point below replaces one third-party library op at the call sites
 * cited (paths relative to the reference checkout).  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions (SURVEY.md section 8b):
 *   - every pointer is a DEVICE pointer unless the parameter name ends in `_host`;
 *   - the caller owns every buffer, outputs are caller-allocated, nothing is retained after return;
 *   - `stream` is a `cudaStream_t` passed as `void*`; work is enqueued, never synchronised;
 *   - return value: 0 on success, negative `FR_E*` otherwise; `fr_last_error()` gives the text;
 *   - no exceptions, no global state apart from the thread-local error string;
 *   - dense matrices are fp32 row-major `[rows, d]` with leading dimension `d` (16-byte aligned rows).
 */
#ifndef FOODREC_B200_H
#define FOODREC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FR_OK 0
#define FR_EINVAL (-1)       /* bad argument (null pointer, negative extent, misalignment)          */
#define FR_EUNSUPPORTED (-2) /* shape outside what the kernels are specialised for                  */
#define FR_ECUDA (-3)        /* CUDA runtime error at launch                                        */

#define FR_SPMM_SEG 128 /* largest allowed `seg_len` (nnz per propagation segment, see fr_spmm_plan_*) */

int fr_version(void);
const char *fr_last_error(void);
/* Number of kernels this library has launched in the calling process (for bench.py's `gpu_launches`). */
int64_t fr_launch_count(void);
/* Optional tracing: while enabled every launch is bracketed by CUDA events on its stream;
 * fr_profile_dump synchronises and writes "kernel,launches,total_us" lines into buf. */
int fr_profile_enable(int on);
int fr_profile_dump(char *buf, int64_t cap);

/* ------------------------------------------------------------------------------------------------
 * Propagation: Y = alpha * (S . X) + beta * Z, S in CSR (fp32 values, int32 indices).
 * Replaces `torch.sparse.mm(S, X)` at FoodRec/models/cikm_model.py:187,199, pricai_modelx.py:183,
 * 197,211,223, lightgcn.py:139 and, with the fused `+ beta*Z` / `alpha` epilogue, the
 * `torch.stack(..).mean(1)` layer combine at cikm_model.py:189-190,201-202 (Horner form:
 * mean_l S^l E0 = (E0 + S(E0 + S(...)))/(L+1)).  The backward of `torch.sparse.mm` w.r.t. X is the
 * same call on the CSR of S^T (== S for the symmetric normalised adjacencies).
 *
 * Rows are processed as SEGMENTS of at most `seg_len` (<= FR_SPMM_SEG) nonzeros so that one popular item cannot
 * serialise a warp; rows longer than a segment are reduced deterministically (fixed order) by the
 * last segment to finish.  The segment plan is built once per graph:
 *
 *   fr_spmm_plan_sizes : from `row_ptr_host` compute n_seg, n_long (fold entries of the rows split in >1 segment),
 *                        n_part (partial-row slots of the fold workspace).
 *   fr_spmm_plan_fill  : fill host arrays seg[n_seg*4] ((row, start, len, -1) for a whole row, (slot, start, len, entry)
 *                        for a segment of a long row), long_rows[n_long*4] (first segment within the row, n_parts,
 *                        part_base, row).  Graphs of >= 262 144 rows schedule their long-row segments by relative position
 *                        inside the row (L2 reuse across popular rows; results unchanged).  A row of more than 16 segments folds
 *                        in two levels: ~sqrt(k) child entries (first_seg, n_parts, part_base, -(parent + 1)), contiguous
 *                        and directly followed by their parent entry (first_child, n_children, part_base, row), so the
 *                        serial chain of the last arriver is ~2 sqrt(k) loads instead of k.  The shape depends on the
 *                        row's length only.
 *   The caller uploads both, and provides `partial` (n_part * d floats) and `counters` (n_long int32,
 *   zero-initialised once; the kernel leaves them zero).
 *
 * act: 0 = none, 1 = tanh (applied after `+ bias`), bias: optional [d] (NULL = none).
 * act/bias serve `tanh(GCNConv(x))` at FoodRec/models/schgn.py:29-41 (S = PyG-normalised directed
 * adjacency incl. self loops, X = lin(x)).
 * d must be 32, 64 or 128.
 */
int fr_spmm_plan_sizes(const int32_t *row_ptr_host, int32_t n_rows, int32_t seg_len, int64_t *n_seg,
                       int64_t *n_long, int64_t *n_part);
int fr_spmm_plan_fill(const int32_t *row_ptr_host, int32_t n_rows, int32_t seg_len, int32_t *seg_host,
                      int32_t *long_rows_host);
int fr_spmm_csr_f32(const int32_t *seg, int64_t n_seg, const int32_t *long_rows, int64_t n_long,
                    const int32_t *col_idx, const float *val, int32_t d, const float *X, const float *Z,
                    float alpha, float beta, const float *bias, int32_t act, float *Y, float *partial,
                    int32_t *counters, void *stream);

/* Same, with two-segment operands: rows [0, x_split) of X come from X0 and rows >= x_split from X1 (row
 * r of the logical table = X1[r - x_split]); likewise Z0 / Z1 / z_split.  X1 == NULL / Z1 == NULL: single
 * table.  Consumes the reference's `torch.cat((user_w, item_emb))` / `cat((item_w, side_w))` ego tables
 * (cikm_model.py:184,195; pricai_modelx.py:180,192-194,206-208,220) without materialising them. */
int fr_spmm_csr_f32_split(const int32_t *seg, int64_t n_seg, const int32_t *long_rows, int64_t n_long,
                          const int32_t *col_idx, const float *val, int32_t d, const float *X0, const float *X1,
                          int32_t x_split, const float *Z0, const float *Z1, int32_t z_split, float alpha, float beta,
                          const float *bias, int32_t act, float *Y, float *partial, int32_t *counters, void *stream);

/* Backward-pass variant with row-activity masks: x_mask[c] == 0 promises that row c of X is exactly zero (its
 * gather is skipped); y_mask[r] (optional) receives whether output row r has a nonzero.  The gradient of a
 * mini-batch ranking loss touches <= 3 B rows, so the first backward layers gather a small fraction of the
 * table.  Results are bit-identical to the unmasked call. */
int fr_spmm_csr_f32_masked(const int32_t *seg, int64_t n_seg, const int32_t *long_rows, int64_t n_long,
                           const int32_t *col_idx, const float *val, int32_t d, const float *X, const float *Z,
                           float alpha, float beta, float *Y, float *partial, int32_t *counters, const uint8_t *x_mask,
                           uint8_t *y_mask, void *stream);

/* Grouped launch: up to FR_SPMM_MAX_TASKS independent propagations (own graph, own operands, fused `+ beta*Z`) in ONE
 * grid.  CLUSSL's three item-side propagations of a layer (pricai_modelx.py:183,197,211: ingredient, image-cluster and
 * text-cluster graphs) are each too small to fill the GPU; launched together their long-row tails overlap and a training
 * step has 6 propagation launches instead of 14.  `blk_map` (device, int32 [n_blocks][2] = task, block of that task;
 * fr_spmm_task_blocks(n_seg) blocks per task) fixes the order in which the tasks' blocks are scheduled.  Results are
 * bit-identical to the separate fr_spmm_csr_f32_split calls. */
#define FR_SPMM_MAX_TASKS 4
typedef struct fr_spmm_task {
    const int32_t *seg;
    int64_t n_seg;
    const int32_t *long_rows;
    int64_t n_long;
    const int32_t *col_idx;
    const float *val;
    const float *X0, *X1;
    int32_t x_split;
    const float *Z0, *Z1;
    int32_t z_split;
    float alpha, beta;
    float *Y, *partial;
    int32_t *counters;
} fr_spmm_task;
int64_t fr_spmm_task_blocks(int64_t n_seg);
int fr_spmm_csr_f32_grouped(const fr_spmm_task *tasks_host, int32_t n_tasks, int32_t d, const int32_t *blk_map,
                            int64_t n_blocks, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Fused ranking loss on gathered rows: BPR + embedding regulariser, forward and backward.
 * Replaces the gathers, `torch.mul(..).sum(1)`, `BPRLoss` and `EmbLoss` at
 * FoodRec/models/cikm_model.py:255-261,267-279, pricai_modelx.py:252-258,266-274,
 * lightgcn.py:159-175 and FoodRec/common/loss.py:28-34,45-50.
 *
 *   mf  = -(1/B) sum_b log(gamma + sigmoid(<E[u_b], E[io+p_b]> - <E[u_b], E[io+n_b]>))
 *   reg = (1/reg_den) * sum_g sqrt(sum over rows r in group g of |T_g[idx_g[r]]|^2)
 *
 * `emb` is the propagated table [n_rows, d] with users first and items from row `item_off`.
 * Groups: up to FR_MAX_REG_GROUPS (table pointer, int64 index pointer, count) triples (a group of count 0 has norm 0,
 * no gradient, and may pass a NULL index pointer); an index
 * equal to `pad_idx[g]` (>= 0) contributes a zero row (nn.Embedding padding_idx semantics are the
 * caller's: the padding row is stored as zeros in the reference, so pad handling only matters for
 * the backward, where that row must receive no gradient).
 * out[0] = mf, out[1] = reg (un-weighted).  coef[B] receives d mf / d(pos-neg) for the backward,
 * gnorm[n_groups] the group norms.  `ws` is a zeroed workspace of fr_rank_loss_ws_floats() floats; its ticket word is left zero.
 */
#define FR_MAX_REG_GROUPS 6
/* floats the caller must provide (zero-initialised once) as `ws` of fr_rank_loss_fwd */
int64_t fr_rank_loss_ws_floats(void);
int fr_rank_loss_fwd(const float *emb, int32_t d, int64_t item_off, const int64_t *u, const int64_t *p,
                     const int64_t *n, int32_t B, float gamma, int32_t n_groups,
                     const float *const *reg_tab_host, const int64_t *const *reg_idx_host,
                     const int64_t *reg_cnt_host, float reg_den, float *out, float *coef, float *gnorm,
                     float *ws, void *stream);
/* d_emb (zero-initialised [n_rows, d] by the caller) += g_mf * d mf/d emb;
 * d_tab[g] (dense, zero-initialised or accumulating) += g_reg * d reg/d T_g.  g_out = {g_mf, g_reg} on device. */
int fr_rank_loss_bwd(const float *emb, int32_t d, int64_t item_off, const int64_t *u, const int64_t *p,
                     const int64_t *n, int32_t B, const float *coef, const float *g_out, float *d_emb,
                     int32_t n_groups, const float *const *reg_tab_host, const int64_t *const *reg_idx_host,
                     const int64_t *reg_cnt_host, const int64_t *reg_pad_host, float reg_den,
                     const float *gnorm, float *const *d_tab_host, uint8_t *emb_mask /* [n_rows] zeroed, or NULL */,
                     void *stream);

/* The two loss modules in their stand-alone form, for callers that already hold scores / gathered rows
 * (`self.mf_loss(pos_scores, neg_scores)`, `self.reg_loss(u_ego, pos_ego, neg_ego)`: FoodRec/common/loss.py:31-34, 44-50).
 *   fr_bpr_scores_fwd: out[0] = -(1/n) sum_i log(gamma + sigmoid(pos[i] - neg[i])); coef[i] = d out / d pos[i] = -d out / d neg[i].
 *   fr_l2_norm_f32:    out[0] = sqrt(sum_i x[i]^2) (torch.norm(x, p=2) of the flattened tensor).
 * One block each, fixed summation order (bit-reproducible); meant for batch-sized inputs. */
int fr_bpr_scores_fwd(const float *pos, const float *neg, int64_t n, float gamma, float *out, float *coef, void *stream);
int fr_l2_norm_f32(const float *x, int64_t n, float *out, void *stream);

/* Row pointers of a CSR from the row indices of a COO (any order; for a row-major-sorted COO -- what the
 * reference builds, FoodRec/models/cikm_model.py:174-180 -- `col`/`val` are then already in CSR order).
 * row_ptr: int32[n_rows + 1]; scratch: int32[n_rows]. */
int fr_csr_from_coo(const int64_t *coo_rows, int64_t nnz, int32_t n_rows, int32_t *row_ptr, int32_t *scratch,
                    void *stream);

/* out[r] = sum_v tab_v[r], r < rows (`item_emb = ingre[:I] + image[:I] + text[:I]`, pricai_modelx.py:219), and
 * the adjoint d_tab_v[r] = (r < rows ? g[r] : 0) over each table's full height rows_total[v] (slice gradient +
 * zero fill of up to four tables in one launch). */
int fr_sum_rows(const float *const *tab_host, int32_t n_tabs, int32_t d, int64_t rows, float *out, void *stream);
int fr_spread_rows(const float *g, int32_t d, int64_t rows, float *const *d_tab_host, const int64_t *rows_total_host,
                   int32_t n_tabs, int32_t accumulate /* 1: d_tab_v[r] += g[r] for r < rows only */,
                   const uint8_t *src_mask /* row mask of g or NULL (= all active) */,
                   uint8_t *const *mask_host /* per-table row masks to write / OR into, or NULL */, void *stream);

/* Row gather out[r] = tab[idx[r]] and its adjoint d_tab[idx[r]] += g[r] (fp32 atomics).
 * Replaces `E[idx]` indexing at pricai_modelx.py:245-247 and the candidate gathers of
 * `inference_fast` (cikm_model.py:294-302, pricai_modelx.py:278-286). */
int fr_gather_rows(const float *tab, int32_t d, const int64_t *idx, int64_t n, float *out, void *stream);
int fr_scatter_add_rows(const float *g, int32_t d, const int64_t *idx, int64_t n, float *d_tab, void *stream);
/* scores[r] = <U[user[r]], I[item[r]]>  (inference_fast / inference_by_user). */
int fr_pair_scores(const float *user_tab, const float *item_tab, int32_t d, const int64_t *user,
                   const int64_t *item, int64_t n, float *scores, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Distance-correlation contrastive term (CLUSSL's live `cl_loss`).
 * Replaces `PRICAI_ModelX.correlation_distance` (FoodRec/models/pricai_modelx.py:409-437) and the
 * three calls + row gathers at :245-247,263.  V <= 3 views are rows `idx[0..n)` of `tab_host[v]`
 * ([rows_v, d] fp32, d in {32, 64}); P <= 3 pairs (a_p, b_p) index the views.
 *   out[p]  = scale * dcov(a,b) / sqrt(max(dcov(a,a) dcov(b,b), 0) + 1e-10),  out[P] = sum_p out[p]
 *             (scale = CLUSSL's `loss_cl`, so `loss_cl * (dcor + dcor + dcor)` costs no extra launch),
 *   dcov(x,y) = sqrt(max(sum(A_x o A_y) / n^2, 0) + 1e-8), A = double-centred
 *   sqrt(max(r_i - 2 x_i.x_j + r_j, 0) + 1e-8).
 * Caller-provided state kept for the backward: Dm [V, n, n], rowmean [V, n], dfds [3 P], gm [V];
 * `ws`: zero-initialised once, fr_dcor_ws_floats(n) floats.
 * Backward: d_tab_host[v] (dense [rows_v, d], may be NULL to skip a view, may alias between views)
 * += sum_p g_out[p] * d out[p] / d tab_v  via fp32 atomics. */
int64_t fr_dcor_ws_floats(int32_t n);
int fr_dcor_fwd(const float *const *tab_host, int32_t V, int32_t d, const int64_t *idx, int32_t n,
                const int32_t *pairs_host, int32_t P, float scale, float *Dm, float *rowmean, float *out /* [P + 1] */,
                float *dfds, float *gm, float *ws, void *stream);
int fr_dcor_bwd(const float *const *tab_host, int32_t V, int32_t d, const int64_t *idx, int32_t n,
                const int32_t *pairs_host, int32_t P, const float *Dm, const float *rowmean,
                const float *dfds, const float *gm, const float *g_out, float *const *d_tab_host,
                uint8_t *const *mask_host /* optional: mark the rows idx[] of each table's mask */,
                float *ws /* fr_dcor_bwd_ws_floats(n) floats of scratch, 16-byte aligned */, void *stream);
int64_t fr_dcor_bwd_ws_floats(int32_t n);

/* ------------------------------------------------------------------------------------------------
 * Ranking: scores = scale * A . B^T + bias  ->  per-row top-k, never materialising [M, N].
 * bf16 tcgen05 GEMM (fp32 accumulate in TMEM) with the top-k selection fused into the epilogue.
 * Replaces, for the dot-product models, `full_sort_predict` + `torch.topk(scores, max(topk))` in
 * `Trainer.evaluate` (FoodRec/common/trainer.py:489-497; SURVEY.md D2/D4), `build_sim` +
 * `torch.topk(adj, k)` of the kNN utilities (FoodRec/utils/utils.py:118-121,132-136,170-172) and
 * the per-item `argsort(|x - c|)[:10][:6]` loop of dataset_process/allrecipes_kmeans.ipynb
 * (argmin |x - c|^2 = argmax x.c - |c|^2 / 2 : bias = -|c|^2 / 2).
 *   A [M, K], B [N, K]: bf16 row-major, K % 8 == 0, 16-byte aligned (fr_f32_to_bf16 converts and
 *   optionally L2-normalises rows as `build_sim` does).
 *   History mask (optional, all three or none): row m is user `row_ids[m]`; columns
 *   `hist_idx[hist_ptr[u] .. hist_ptr[u+1])` (sorted ascending) are excluded -- MMRec's
 *   `scores[train items] = -inf`; the reference applies no mask (SURVEY.md D1) = pass NULLs.
 *   out_val / out_idx [M, topk] (topk <= 64), descending, ties to the lower column, -1 / -inf padding.
 * fr_rescore_topk_f32 re-scores the kc >= k bf16 candidates exactly in fp32 (A_f32 rows `a_rows[m]` or m) and keeps
 * the best k; out_idx is int64 (`idx64` != 0, like `torch.topk`) or int32.  metric 1 ranks by exact squared
 * distance.  With `cert` != NULL it also writes a per-row CERTIFICATE: cert[m] = 1 iff no column outside the
 * candidate set can belong to the fp32 top-k, i.e. fewer than kc eligible columns existed or
 *   cand_val[m, kc-1] + |scale| (|a' - a| max|b'| + |a| max|b' - b| + K 2^-23 |a'| max|b'|)  <  (k-th best fp32 re-score)
 * with a' = bf16(A_m), b' = bf16(B_n) (`cand_val` = the bf16-pass scores of the candidates, `bmax` = the two
 * device floats {max_n |b'_n|, max_n |b'_n - B_n|} from fr_max_row_norm).  Rows with
 * cert = 0 are re-ranked by the caller with a wider candidate set or by fr_exact_topk_f32.
 * fr_exact_topk_f32 is the exact path for such rows: fp32 scores of rows A[a_rows[0..Mf)] against ALL N columns on
 * the CUDA cores (scores_ws: Mf * N floats of scratch), optional history mask (`hist_rows[r]` = CSR row of result
 * row r), radix select of the k best, ordered by (score desc, column asc); -1 / -inf padding. */
int fr_f32_to_bf16(const float *x, void *y_bf16, int64_t rows, int32_t d, int32_t l2_normalise, void *stream);
int64_t fr_gemm_topk_ws_bytes(int32_t M); /* caller-provided scratch (candidate lists, L2-resident) */
int fr_gemm_topk_bf16(const void *A_bf16, int32_t M, const void *B_bf16, int32_t N, int32_t K, float scale,
                      const float *bias, const int64_t *row_ids, const int64_t *hist_ptr, const int32_t *hist_idx,
                      int32_t topk, float *out_val, int32_t *out_idx, void *ws, int64_t ws_bytes, void *stream);
int fr_max_row_norm(const float *B, int64_t rows, int32_t d, float *out /* 2 device floats */, void *stream);
int fr_rescore_topk_f32(const float *A, const int64_t *a_rows, const float *B, int32_t d, float scale,
                        const float *bias, int32_t metric /* 0: scale*a.b+bias, 1: -|a-b|^2 */, const int32_t *cand,
                        const float *cand_val, int32_t kc, int32_t M, int32_t k, float *out_val, void *out_idx,
                        int32_t idx64, const float *bmax, uint8_t *cert, void *stream);
int fr_exact_topk_f32(const float *A, const int64_t *a_rows, int32_t Mf, const float *B, int32_t N, int32_t d,
                      float scale, const float *bias, int32_t metric, const int64_t *hist_rows,
                      const int64_t *hist_ptr, const int32_t *hist_idx, int32_t k, float *scores_ws, float *out_val,
                      int64_t *out_idx, void *stream);
/* The same rows with a per-row THRESHOLD: `thr[r]` is a lower bound of row r's k-th best fp32 score (the caller has it
 * from the re-scored candidates, minus a rounding margin), so only columns scoring >= thr[r] can belong to the result.
 * Nothing dense is written: the SIMT fp32 scoring pass appends the few qualifying (score, column) pairs to a per-row
 * list (history columns dropped by binary search) and one CTA per row sorts its list (score desc, column asc).
 * ws: fr_exact_topk_thr_ws_bytes(Mf) bytes, 8-byte aligned.  *overflow (device int) = rows whose list did not fit
 * (massive ties): their outputs are untouched and the caller re-runs them with fr_exact_topk_f32. */
int64_t fr_exact_topk_thr_ws_bytes(int32_t Mf);
int fr_exact_topk_thr_f32(const float *A, const int64_t *a_rows, int32_t Mf, const float *B, int32_t N, int32_t d,
                          float scale, const float *bias, int32_t metric, const int64_t *hist_rows,
                          const int64_t *hist_ptr, const int32_t *hist_idx, int32_t k, const float *thr, void *ws,
                          float *out_val, int64_t *out_idx, int32_t *overflow, void *stream);

/* Mean cosine similarity of dense rows A[i] with gathered rows T[idx[i]] (eps = 1e-8 on each norm):
 * HealthRec's knowledge-distillation term `1 - cosine_similarity(item_know, cat(pos_e, neg_e)).mean()`
 * (FoodRec/models/cikm_model.py:263-264).  cosv / na / nt [n] keep the per-row state for the backward, which
 * writes dA [n, d] (or NULL) and scatter-adds into the dense dT (or NULL). */
int fr_cosine_mean_fwd(const float *A, const float *T, const int64_t *idx, int64_t n, int32_t d, float *out, float *cosv,
                       float *na, float *nt, void *stream);
int fr_cosine_mean_bwd(const float *A, const float *T, const int64_t *idx, int64_t n, int32_t d, const float *cosv,
                       const float *na, const float *nt, const float *g_out, float *dA, float *dT, void *stream);

/* ------------------------------------------------------------------------------------------------
 * SimCLR NT-Xent ("InfoNCE") over the two halves of hidden [2b, d] (d in {32, 64}).
 * Replaces `PRICAI_ModelX.CL_loss` (FoodRec/models/pricai_modelx.py:354-378; dormant in the reference, its
 * call is commented out at :259): cosine-normalise (optional), logits / temperature, diagonal of the aa / bb
 * blocks masked, two cross-entropies, (loss_a + loss_b) / b.  Equivalent single-Gram form:
 *   out[0] = sum_r [ logsumexp_{c != r} G[r, c] - G[r, pair(r)] ] / b^2,  G = Hn Hn^T / temperature.
 * State for the backward (caller-allocated): hn [2b, d], norm [2b], G [2b, 2b], lse [2b];
 * ws: fr_infonce_ws_floats(2b) floats of scratch.  d_hidden [2b, d] is written (not accumulated). */
int64_t fr_infonce_ws_floats(int32_t n);
int fr_infonce_fwd(const float *hidden, int32_t b, int32_t d, float temperature, int32_t normalise, float *hn,
                   float *norm, float *G, float *lse, float *out, float *ws, void *stream);
int fr_infonce_bwd(const float *hn, const float *norm, const float *G, const float *lse, int32_t b, int32_t d,
                   float temperature, int32_t normalise, const float *g_out, float *d_hidden, void *stream);

/* ------------------------------------------------------------------------------------------------
 * SCHGN per-pair scorer for full-sort evaluation (d = 64).
 * Replaces `SCHGN.full_sort_predict` -> `compute_score` (FoodRec/models/schgn.py:318-345, 233-268) with the
 * two attention levels (:159-184, :186-206) fused; the reference builds python lists over every item,
 * re-uploads the [I, Dv] image matrix and runs the GCN once PER USER.  The caller precomputes what does not
 * depend on the user (final rows = table + GCN row; "key" = image of a row under the matching slice of
 * W_att_ingre / W_att_comp):
 *   ingre_key / ingre_final / ingre_comp [G + 1, 64]  per ingredient code (code G = padding, all-zero final row)
 *   img_key [I, 64]        img_emb W_att_ingre[:, image]^T + b_att_ingre
 *   comps / comp_keys [I, 3, 64]   item, image, health final rows and their W_att_comp[:, component] images
 *   user_key / user_comp / user_hidden / user_final [nu, 64]   per user of the batch (biases folded in)
 * fr_schgn_attend writes att [nu, I, 64] (attended ingredient row) and logits [nu, 4, I] (component logits in
 * the reference order item, ingredients, image, health); fr_schgn_score applies the component softmax over the
 * reference's `.view(b, -1)` grouping of those logits (schgn.py:198 -- row r reads flat entries 4r .. 4r+3 of
 * the [4, I] block), then relu(W_concat [u; x; u * x] + b) . output_mlp, and writes scores [nu, I].
 * tanh(a + b) is evaluated as 1 - 2 / (1 + e^{2a} e^{2b}) with the factors shared across users / items (precise
 * expf, Newton-refined reciprocal; |error| ~ 2e-7, the order of tanhf's own). */
int fr_schgn_attend(const float *user_key, const float *user_comp, int32_t nu, const int32_t *codes, int32_t slots,
                    const int32_t *nums, int32_t n_items, const float *ingre_key, const float *ingre_final,
                    const float *ingre_comp, const float *img_key, const float *comp_keys, const float *h_ingre,
                    const float *h_comp, int32_t d, float *att, float *logits, void *stream);
int fr_schgn_score(const float *user_final, const float *user_hidden, int32_t nu, const float *W_item,
                   const float *W_prod, const float *w_out, const float *comps, const float *att, const float *logits,
                   int32_t n_items, int32_t d, float *scores, void *stream);
/* fr_schgn_score with the row-wise top-k fused in: the [nu, I] score block never reaches HBM.  Each CTA keeps the k best
 * of its 256 items (bitonic sort in shared memory; `user_ids[nu]` + the sorted history CSR exclude each user's training
 * items, NULL = no mask as in the reference, trainer.py:495-497), a second launch merges the block winners per user.
 * Output: out_val / out_idx [nu, k], score descending, ties to the lower item; -inf / -1 when fewer than k items remain.
 * ws: fr_schgn_score_topk_ws_bytes(nu, n_items, k) bytes, 8-byte aligned.  k <= 64. */
int64_t fr_schgn_score_topk_ws_bytes(int32_t nu, int32_t n_items, int32_t k);
int fr_schgn_score_topk(const float *user_final, const float *user_hidden, int32_t nu, const float *W_item,
                        const float *W_prod, const float *w_out, const float *comps, const float *att, const float *logits,
                        int32_t n_items, int32_t d, const int64_t *user_ids, const int64_t *hist_ptr,
                        const int32_t *hist_idx, int32_t k, void *ws, float *out_val, int64_t *out_idx, void *stream);
/* The same scorer over per-user candidate lists (by-user evaluation, FoodRec/common/trainer.py:231-282: each user's
 * held-out positives, then sampled negatives, scored as ONE `inference_by_user` batch).  User u of the call owns pairs
 * q = ptr[u] - ptr[0] .. ptr[u+1] - ptr[0] - 1 (ptr int64 [nu + 1], strictly increasing: no empty list; n_pairs =
 * ptr[nu] - ptr[0]); pair q is candidate items[q] (int32).  The component softmax groups each list's own logits as the
 * reference does with b = L, the list length: row r takes flat entries 4r .. 4r+3 of the list's component-major [4, L]
 * block, so it depends on the list's order and length.  Item-side tables as above, user rows [nu, 64].
 *   fr_schgn_attend_pairs: att [n_pairs, 64] and logits [4 n_pairs] (list of user u at 4 (ptr[u] - ptr[0]), [4, L]).
 *     Groups the pairs by item on the device (ws: fr_schgn_attend_pairs_ws_bytes(nu, n_pairs, n_items) bytes,
 *     16-byte aligned).  The lists are checked on the device: *status (device int32, zeroed by the caller) gets
 *     FR_PAIRS_BAD_PTR when a list is empty, ptr does not increase or ptr[nu] - ptr[0] != n_pairs, and
 *     FR_PAIRS_BAD_ITEM for an item outside [0, n_items).  Bad lists / pairs are skipped, never dereferenced; their
 *     outputs are undefined, so the caller reads *status before it uses any score.  A bad ptr can make the lists that
 *     pass their own check overlap, so once FR_PAIRS_BAD_PTR is set nothing after the check is computed: att and
 *     logits are left as they were and no byte past the workspace's grp array is written.
 *   fr_schgn_score_pairs: scores [n_pairs] from the att / logits of fr_schgn_attend_pairs on the same ptr / items.
 * Float tables 16-byte aligned; at most 2^31 - 1 pairs per call. */
#define FR_PAIRS_BAD_PTR 1
#define FR_PAIRS_BAD_ITEM 2
int64_t fr_schgn_attend_pairs_ws_bytes(int32_t nu, int64_t n_pairs, int32_t n_items);
int fr_schgn_attend_pairs(const float *user_key, const float *user_comp, int32_t nu, const int64_t *ptr,
                          const int32_t *items, int64_t n_pairs, const int32_t *codes, int32_t slots, const int32_t *nums,
                          int32_t n_items, const float *ingre_key, const float *ingre_final, const float *ingre_comp,
                          const float *img_key, const float *comp_keys, const float *h_ingre, const float *h_comp,
                          int32_t d, void *ws, int64_t ws_bytes, float *att, float *logits, int32_t *status,
                          void *stream);
int fr_schgn_score_pairs(const float *user_final, const float *user_hidden, int32_t nu, const int64_t *ptr,
                         const int32_t *items, int64_t n_pairs, const float *W_item, const float *W_prod,
                         const float *w_out, const float *comps, const float *att, const float *logits, int32_t n_items,
                         int32_t d, float *scores, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Row-partitioned multi-GPU propagation over peer memory (one process per GPU, one NVLink/NVSwitch node).
 * The reference is single-GPU (SURVEY.md 8e); the baseline exchange is one NCCL all-gather per layer
 * (dist.py).  Here the all-gather of layer l+1's input is fused into layer l's kernel: the push epilogue
 * stores every finished output row at row `row_off + r` of `n_peers` (<= 8) full-size tables, one per rank,
 * mapped with CUDA IPC.  Y may be NULL (only the pushed copies are wanted).  Ranks order themselves with the
 * caller's stream-ordered barrier; no kernel waits on another rank.
 *   fr_peer_alloc   cudaMalloc (zeroed) + 64-byte IPC handle to send to the other ranks
 *   fr_peer_open    map another rank's table from its handle;  fr_peer_close / fr_peer_free  undo the two
 *   fr_push_rows    the same exchange for rows no SpMM produced (the layer-0 input) */
/* The exchange as NCCL collectives behind this ABI (SURVEY.md 8b: `fr_allgather_rows`).  NCCL is bound at run time
 * (dlopen of the libnccl.so.2 the process has loaded -- PyTorch links it; FR_NCCL_LIBRARY overrides), so the library has no
 * link-time NCCL dependency.  One communicator per process (= per GPU), created from a 128-byte unique id that rank 0
 * obtains and the caller distributes (dist.RowComm sends it through torch.distributed):
 *   fr_comm_unique_id       rank 0: ncclGetUniqueId -> id128
 *   fr_comm_init            every rank, on its current device: ncclCommInitRank -> *comm;  fr_comm_destroy undoes it
 *   fr_allgather_rows       x_full[world * rows_per_rank, d] <- every rank's x_local[rows_per_rank, d], on `stream`
 *   fr_reduce_scatter_rows  g_local[rows_per_rank, d] <- sum over ranks of block `rank` of their g_full (the adjoint)
 *   fr_comm_version         NCCL version code, 0 when NCCL cannot be bound */
int fr_comm_version(void);
int fr_comm_unique_id(void *id128);
int fr_comm_init(const void *id128, int32_t rank, int32_t world, void **comm);
int fr_comm_destroy(void *comm);
int fr_allgather_rows(void *comm, const float *x_local, int64_t rows_per_rank, int32_t d, float *x_full, void *stream);
int fr_reduce_scatter_rows(void *comm, const float *g_full, int64_t rows_per_rank, int32_t d, float *g_local, void *stream);
int fr_peer_alloc(int64_t bytes, void **ptr, void *handle64);
int fr_peer_open(const void *handle64, void **ptr);
int fr_peer_close(void *ptr);
int fr_peer_free(void *ptr);
int fr_push_rows(const float *src, int64_t rows, int32_t d, float *const *peers_host, int32_t n_peers, int64_t row_off,
                 void *stream);
int fr_spmm_csr_f32_push(const int32_t *seg, int64_t n_seg, const int32_t *long_rows, int64_t n_long,
                         const int32_t *col_idx, const float *val, int32_t d, const float *X, const float *Z, float alpha,
                         float beta, float *Y, float *partial, int32_t *counters, float *const *peers_host,
                         int32_t n_peers, int64_t row_off, void *stream);

/* Dense Adam over many tensors in one launch (plus a one-thread prologue that advances the device-side step counter
 * and derives the bias corrections, so the pair replays inside a CUDA graph).  `lr` is a kernel argument here, fixed
 * at capture; fr_optim_step below reads it from the device instead.  Replaces `optim.Adam(...).step()` of
 * FoodRec/common/trainer.py:144,205 with torch.optim.Adam's arithmetic (amsgrad = False, weight_decay = 0); dense on
 * purpose: rows with a zero gradient still move while their first moment decays.  HealthRec's trainable raw-feature
 * tables (cikm_model.py:83,87) make this the largest HBM stream of its step.
 * Hyper-parameters are doubles like torch's python floats: `1 - beta` is formed in double and then rounded to fp32.
 *   step_dev    device int32, the number of steps taken so far (incremented once per call)
 *   scalars_dev device float[2] scratch
 * More than FR_ADAM_MAX_TENSORS non-empty tensors take several launches, each tensor exactly one; zero-size tensors
 * are skipped.  Every tensor is validated before the first launch, so a rejected call changes nothing. */
#define FR_ADAM_MAX_TENSORS 64
typedef struct fr_adam_tensor {
    float *param;
    const float *grad;
    float *exp_avg;
    float *exp_avg_sq;
    int64_t n;
} fr_adam_tensor;
int fr_adam_step(const fr_adam_tensor *tensors_host, int32_t n_tensors, double lr, double beta1, double beta2, double eps,
                 int32_t *step_dev, float *scalars_dev, void *stream);

/* The learners of the reference trainer's optimizer factory (FoodRec/common/trainer.py:137-154: Adam, SGD, Adagrad,
 * RMSprop with `lr` and `weight_decay`, every other option at torch's default) on the same multi-tensor launches as
 * fr_adam_step, which runs the FR_OPTIM_ADAM rule of this entry point.  Arithmetic and its order follow torch 2.11's
 * `_single_tensor_*` functions; with wd != 0 the gradient is first replaced by g' = g + wd p (torch's L2 term, not
 * AdamW's decoupled decay):
 *   FR_OPTIM_ADAM     state0 = exp_avg, state1 = exp_avg_sq, step_dev   fr_adam_step's update on g'     28 B / param
 *   FR_OPTIM_SGD      no state (momentum 0)                             p += (-lr) g'                    12 B / param
 *   FR_OPTIM_ADAGRAD  state0 = sum, step_dev (lr_decay 0)               s += g' g'; p += (-lr) g' / (sqrt(s) + eps)
 *   FR_OPTIM_RMSPROP  state0 = square_avg (momentum 0, not centred)     a = a alpha + ((1 - alpha) g') g';
 *                                                                       p += (-lr) g' / (sqrt(a) + eps)  20 B / param
 * (Adagrad moves 20 B / param too.)  Unused state pointers of a rule may be NULL.
 *   lr_dev      device double: the learning rate, read by the one-thread prologue of every call, so a call captured
 *               in a CUDA graph uses the value the scalar holds at each replay.  A negative or NaN value is rejected
 *               there: the call then changes no parameter, no state and no step, and leaves scalars_dev[0] = NaN.
 *   step_dev    device int32, incremented once per call; required by Adam and Adagrad, may be NULL otherwise
 *   scalars_dev device float[2] scratch
 * Host-side rejections (unknown rule, negative eps / weight_decay, betas or alpha out of range, a NULL pointer the
 * rule needs, a negative extent) happen before anything is launched, so they change nothing either.  Batching into
 * launches of at most FR_ADAM_MAX_TENSORS non-empty tensors is that of fr_adam_step. */
#define FR_OPTIM_ADAM 0
#define FR_OPTIM_SGD 1
#define FR_OPTIM_ADAGRAD 2
#define FR_OPTIM_RMSPROP 3
typedef struct fr_optim_tensor {
    float *param;
    const float *grad;
    float *state0;
    float *state1;
    int64_t n;
} fr_optim_tensor;
typedef struct fr_optim_hyper {
    double beta1, beta2;  /* Adam: betas, each in [0, 1)                   */
    double alpha;         /* RMSprop: smoothing constant, >= 0             */
    double eps;           /* Adam, Adagrad, RMSprop: >= 0                  */
    double weight_decay;  /* every rule: >= 0                              */
} fr_optim_hyper;
int fr_optim_step(int32_t rule, const fr_optim_tensor *tensors_host, int32_t n_tensors, const fr_optim_hyper *hyper,
                  const double *lr_dev, int32_t *step_dev, float *scalars_dev, void *stream);

/* Measurement probe (not on the product path): gathers `n_idx` rows of a d = 64 table and does nothing else;
 * its bytes/s is the gather roofline the propagation kernel is compared with (scripts/microbench_gather_roofline.py).
 * out: blocks * 32 floats of scratch. */
int fr_probe_gather(const float *tab, int32_t d, const int32_t *idx, int64_t n_idx, int32_t inflight, int32_t blocks,
                    float *out, void *stream);

/* Negative sampling on the device: out_neg[i] = an item drawn uniformly from the items NOT in users[i]'s sorted
 * exclusion list (CSR over users: training + validation/test items).  Replaces the per-sample python rejection loop
 * `TrainDataLoader.get_random_neg` (FoodRec/utils/dataloader.py:145-151).  Counter-based generator: the result is a
 * pure function of (seed, step, i); same distribution as the reference, not numpy's stream.  *fail_count is
 * incremented for a sample whose user excludes (almost) everything (4096 rejected draws); the caller checks it. */
int fr_sample_negatives(const int64_t *excl_ptr, const int32_t *excl_idx, const int64_t *users, int64_t n,
                        int32_t n_items, uint64_t seed, uint64_t step, int64_t *out_neg, int32_t *fail_count,
                        void *stream);

/* ------------------------------------------------------------------------------------------------
 * Evaluation metrics on the device (the host step after full-sort / by-user ranking: metrics.topk_metrics and
 * metrics.by_user_metrics, FoodRec/utils/topk_evaluator.py:68-115, FoodRec/common/matrics.py:9-102,
 * FoodRec/common/trainer.py:49-69,231-282).  Both write SUMS over users in fp64 (the caller divides); per-user values
 * are optional.  Block partials are folded by the last block in a fixed order: bit-reproducible on a given device.
 * `ws`: fr_eval_metrics_ws_bytes() bytes, 16-byte aligned, zeroed once; its ticket word is left zero, so the
 * launches replay inside a CUDA graph.  One `ws` serves both entry points, one launch at a time.
 *
 * fr_topk_metrics: top [n, K] (int32, or int64 with idx64 != 0; K <= 64; entries < 0 are padding, never a hit) against
 * the held-out positives pos_idx[pos_ptr[r] .. pos_ptr[r+1]) (sorted, unique per row), pos_len[r] = the length of the
 * list as given (duplicates included: the host divides by it); cutoffs c_i in 1..K.  A repeated column counts as a hit
 * each time.  disc / ideal [K] fp32: 1 / log2(rank + 1) and its running sum, computed by the caller with numpy's
 * expressions (metrics._ndcg_tables).  Per user and cutoff c, with cum = hits in the first c columns:
 *   recall = cum / pos_len, precision = cum / c (fp64); recall2 contributes cum (its mean = sum cum / sum pos_len);
 *   ndcg = (fp32 running sum of disc over the hit columns) / ideal[min(c, pos_len) - 1] (fp32);
 *   map = fp32( (sum over hit columns j < c of cum_j / (j + 1), fp64) / min(c, pos_len) ).
 * These are bit-identical to the host's per-user values.  sums: [FR_TOPK_METRICS][n_cut] in the order recall, recall2,
 * ndcg, precision, map, then sum pos_len.  per_user (or NULL): [n][FR_TOPK_METRICS][n_cut] fp64.  pos_len < 1 gives NaN.
 *
 * fr_by_user_metrics: user r owns scores[ptr[r] .. ptr[r+1]), its first n_pos[r] entries are the positives.  Per user:
 *   AUC = #{(i positive, j negative) : s_j < s_i} / (n_pos * neg_num)   (neg_num as given, like the reference);
 *   rank_i = #{j : s_j > s_i} + #{j > i : s_j == s_i}, the position of i in np.argsort(s, kind="stable")[::-1] --
 *   the host's default (unstable) argsort agrees with it wherever a positive's score ties no other score;
 *   Recall@c = #{i : rank_i < c} / n_pos, NDCG@c = sum_{rank_i < c} 1/log2(rank_i + 2) / sum_{t < min(c, L, n_pos)}
 *   1/log2(t + 2) (fp64, L = segment length).  Cutoffs 1..64.  sums: [AUC, Recall@c_0.., NDCG@c_0..]; per_user (or
 *   NULL): [n][1 + 2 n_cut] fp64.  A user with n_pos < 1 or n_pos > L gives NaN.
 */
#define FR_EVAL_MAX_CUTOFFS 8
#define FR_TOPK_METRICS 5
int64_t fr_eval_metrics_ws_bytes(void);
int fr_topk_metrics(const void *top, int32_t idx64, int64_t n, int32_t K, const int64_t *pos_ptr, const int32_t *pos_idx,
                    const int32_t *pos_len, const int32_t *cutoffs_host, int32_t n_cut, const float *disc,
                    const float *ideal, double *sums, double *per_user, void *ws, void *stream);
int fr_by_user_metrics(const float *scores, const int64_t *ptr, const int32_t *n_pos, int64_t n, int32_t neg_num,
                       const int32_t *cutoffs_host, int32_t n_cut, double *sums, double *per_user, void *ws,
                       void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FOODREC_B200_H */
