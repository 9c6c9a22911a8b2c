/* libwmf_b200.so - C ABI of the B200-native WMF (implicit-feedback ALS) train + top-N path.
 *
 * The reference (titoeb/RecModel) has no FFI, plugin or operator registry on this path: the
 * whole of WMF is NumPy/SciPy Python (RecModel/wmf_model.py:1-6, SURVEY.md D2). The drop-in
 * boundary is therefore the Python class `WMF`; these entry points are what a maintainer would
 * bind from that class with ctypes (see INTEGRATION.md), one per NumPy/LAPACK call site the
 * kernels replace. Each declaration cites the reference lines it stands in for, relative to
 * /root/reference/.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer unless the name ends in _host. The caller owns every
 *    buffer; the library allocates nothing persistent.
 *  - `stream` is a cudaStream_t passed as void*. All work is stream-ordered, no hidden syncs.
 *  - Factor matrices are row-major float32 with leading dimension ld (elements).
 *  - CSR: indptr int64[rows+1], indices int32[nnz], data float32[nnz].
 *  - Return 0 on success; non-zero = error, text from wmf_last_error() (thread-local).
 *  - sm_100a only. There is no CPU path: on a machine without a B200-class device every
 *    compute entry point returns WMF_ERR_NO_DEVICE.
 */
#ifndef WMF_B200_H
#define WMF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WMF_OK 0
#define WMF_ERR_INVALID 1     /* bad argument (null pointer, f out of range, ...) */
#define WMF_ERR_WORKSPACE 2   /* workspace too small: ask wmf_*_workspace_bytes */
#define WMF_ERR_CUDA 3        /* CUDA runtime error, see wmf_last_error */
#define WMF_ERR_NO_DEVICE 4   /* no sm_100 device visible */
#define WMF_ERR_UNSUPPORTED 5 /* shape outside what the selected algorithm handles */

#define WMF_MAX_F 320 /* largest factor width (dim, +1 with bias) any kernel accepts */

/* Half-step algorithm selector */
#define WMF_ALGO_AUTO 0
#define WMF_ALGO_SIMT 1    /* FP32 CUDA-core Gram + Cholesky/LU; any f <= WMF_MAX_F; accuracy cross-check */
#define WMF_ALGO_TCGEN05 2 /* whitened factors, FP16-split tcgen05 Gram, conjugate gradients on the matrix in TMEM; f <= 256, biases included */
#define WMF_ALGO_TCGEN05_DIRECT 3 /* same pipeline, every system factorised (block Gauss-Jordan in TMEM): the fallback of 2, selectable as a cross-check */

/* Count preprocessing modes */
#define WMF_PREPROCESS_LOG 0    /* d = alpha*log(1+beta*x)   wmf_model.py:120 */
#define WMF_PREPROCESS_LINEAR 1 /* d = alpha*x               wmf_model.py:123 */

const char* wmf_last_error(void);
int wmf_version(void);
/* Kernel launches this library has issued in this process so far (launch sites counted where they are
 * issued; replays of a captured CUDA graph are not seen here: multiply the count of the capture). */
long long wmf_launch_count(void);
/* 0 if a usable sm_100 device is current, else WMF_ERR_NO_DEVICE. Fills sm_count if non-null. */
int wmf_device_check(int* sm_count);

/* K6. In-place count preprocessing.                      replaces wmf_model.py:66-70,119-123 */
int wmf_preprocess(float* data, int64_t nnz, int mode, float alpha, float beta, void* stream);

/* N1. CSR of the transpose, on the device:             replaces count_mat.T.tocsr() (wmf_model.py:128).
 * A stable radix sort of the entries by column: every output row holds ascending original row ids (SciPy's
 * order), whatever the column order inside the input rows; duplicate entries are kept. Transposing twice
 * canonicalises a matrix (sorted indices). out_indptr int64[cols+1], out_indices int32[nnz], out_data float[nnz]. */
size_t wmf_csr_transpose_workspace_bytes(int64_t rows, int64_t cols, int64_t nnz);
int wmf_csr_transpose(const int64_t* indptr, const int32_t* indices, const float* data, int64_t rows, int64_t cols,
                      int64_t nnz, int64_t* out_indptr, int32_t* out_indices, float* out_data, void* ws,
                      size_t ws_bytes, void* stream);

/* K1. G = Y^T Y + lambda*I  (f x f, row-major, ld = f).  replaces np.dot(Y.T,Y)+lambda*eye at
 * wmf_model.py:215,244,258,332 (and the Gram inside :85,:88). ones_col0 != 0 computes with
 * column 0 of Y replaced by 1 (the bias path's Y[:,0] = 1, :331) without touching Y.
 * Deterministic: per-CTA partials in `ws`, reduced in a fixed order. */
size_t wmf_gram_workspace_bytes(int64_t n, int f);
int wmf_gram(const float* Y, int64_t n, int f, int64_t ldy, float lambda, int ones_col0,
             float* G, void* ws, size_t ws_bytes, void* stream);
/* The same Gram in two stages, for row-sharded runs (SURVEY.md 8e). The n rows are cut into
 * wmf_gram_blocks(n) blocks of wmf_gram_block_rows(n) rows (a function of n alone). wmf_gram_partials
 * writes the double-precision partial of every block of the local slice Y[0, nloc) = global rows
 * [row0, row0 + nloc) into `partials` (wmf_gram_workspace_bytes(n, f) bytes, block b at offset b*f*f doubles;
 * row0 and nloc must be whole blocks, the last block of the matrix may be short). After the ranks have
 * exchanged their blocks (blocks a rank does not own zero-filled, then one sum all-reduce: x + 0 is exact),
 * wmf_gram_reduce adds all blocks in block order and rounds once: the same bits on every rank and the same
 * bits wmf_gram gives on one GPU. */
int64_t wmf_gram_block_rows(int64_t n);
int64_t wmf_gram_blocks(int64_t n);
int wmf_gram_partials(const float* Y, int64_t row0, int64_t nloc, int64_t n, int f, int64_t ldy, int ones_col0,
                      void* partials, size_t partials_bytes, void* stream);
int wmf_gram_reduce(const void* partials, int64_t n, int f, float lambda, float* G, void* stream);

/* Exchange step of a row-sharded half-step over peer memory (SURVEY.md 8e; replaces an NCCL all-gather of the
 * new factor shard and an all-reduce of Gram block partials). Copies `bytes` bytes at `src` (local memory) to byte
 * offset dst_offset_bytes of each of `world` buffers whose PEER-MAPPED base addresses are in the device table
 * peer_bases_dev[world] (symmetric allocations, e.g. torch.distributed._symmetric_memory buffer_ptrs); rank `self`
 * (-1: none) is skipped because the source already lives in its copy. Stores go over NVLink as posted writes; the
 * caller orders them before the readers with one cross-rank barrier per half-step. */
int wmf_peer_broadcast(const void* src, size_t bytes, const void* const* peer_bases_dev, int world, int self,
                       size_t dst_offset_bytes, void* stream);

/* K2. One ALS half-step over `rows` CSR rows:            replaces the row loops at
 * wmf_model.py:220-239 (recompute_factors), :337-350 (recompute_factors_bias) and the Pool
 * variants :242-309.
 *   x_r = (G + sum_j d_j y_j y_j^T)^-1  sum_j (d_j+1) y_j ,   j over the stored entries of row r
 * Y has `cols` rows (the columns of the count matrix). bias != 0: y_j has column 0 replaced by 1 and
 * d_j = data_j - Y[j*ldy+0] (:328-343); G must then come from wmf_gram(..., ones_col0=1). Rows with no
 * entries give the zero vector (:223-225; with bias solve(G,0)=0 is the same). `row_order` (nullable) is
 * the processing schedule: int32[order_len] holding every row id of [0,rows) exactly once plus any number
 * of -1 padding slots. The persistent CTAs deal its entries out round-robin (slot s goes to CTA
 * s mod gridDim on the tcgen05 path, to the next free CTA on the SIMT path), so a schedule
 * built with longest rows first balances the power-law tail; it never changes a row's arithmetic.
 * X row r is written at X + r*ldx.
 *
 * WMF_ALGO_TCGEN05 (f <= 256, with or without biases; WMF_ALGO_AUTO picks it whenever it applies):
 *   G = L L^T in double, Y~ = Y L^-T ("whitened" factors, zero padded to 128 or 256 columns), then per row
 *   (I + sum_j d_j y~_j y~_j^T) x' = sum_j (d_j+1) y~_j on the tensor cores and x = L^-T x'. The whitened
 *   matrix has its spectrum in [1, ~10], which makes the FP16-split tcgen05 Gram + in-TMEM Gauss-Jordan
 *   accurate to ~1e-6 of the fp64 solution. Rows with at most wmf_als_dual_max_entries() stored entries solve
 *   the n x n dual system (I + W W^T) u = (d+1)/sqrt(d), W = sqrt(d) y~, x' = W^T u instead (any f <= 256);
 *   longer rows solve the f x f system on tcgen05 when f <= 128 and on the CUDA-core kernel above that.
 *   Rows with a negative weight (possible with biases only) are solved by the CUDA-core LU kernel.
 * WMF_ALGO_SIMT: FP32 CUDA-core Gram + Cholesky / LU with partial pivoting in the original variables;
 *   any f <= WMF_MAX_F; accuracy cross-check and the fix-up path of the tcgen05 algorithm. */
size_t wmf_als_half_step_workspace_bytes(int64_t rows, int64_t cols, int f, int algo);
/* 1 if `algo` (WMF_ALGO_SIMT / WMF_ALGO_TCGEN05) handles factor width f with/without bias, else 0. */
int wmf_als_half_step_supports(int algo, int f, int bias);
/* The tcgen05 path cuts rows with more stored entries than this into segments that different CTAs
 * accumulate (partial Grams summed in segment order before the solve: a function of the row alone, so
 * sharding never changes a row's arithmetic). A schedule should cost such a row as that many entries. */
int wmf_als_row_split_entries(void);
/* Rows with at most this many stored entries take the dual (n x n) tcgen05 kernel. */
int wmf_als_dual_max_entries(void);
/* Workspace for a call whose long rows make `segments` segments in total: a row of n > L =
 * wmf_als_row_split_entries() stored entries makes at most ceil(n / L) of them. The plain query above
 * provides scratch for 2048 segments; a row that finds no scratch is accumulated whole by one CTA. */
size_t wmf_als_half_step_workspace_bytes_split(int64_t rows, int64_t cols, int f, int algo, int64_t segments);
int wmf_als_half_step(const int64_t* indptr, const int32_t* indices, const float* data,
                      int64_t rows, int64_t cols, const int32_t* row_order, int64_t order_len, const float* Y,
                      int64_t ldy, int f,
                      const float* G, int bias, float* X, int64_t ldx, int algo, void* ws,
                      size_t ws_bytes, void* stream);
/* Flags of the last tcgen05 call that used `ws` (read after the stream has drained): bit 1 a pivot block
 * failed (row re-solved by the LU kernel), bit 3 G was not positive definite (all rows solved by the LU
 * kernel); *fixup_rows = rows the LU kernel solved. */
int wmf_als_half_step_status(const void* ws, int* flags_host, int* fixup_rows_host, void* stream);
/* *any_row_host = 1 if, in the last WMF_ALGO_TCGEN05 call that used `ws`, the conjugate gradients of some row did not
 * reach the residual bound within their product budget, so that the row was factorised in tensor memory instead (0 on
 * the reference's weightings; weights in the thousands get there). Replaces nothing in the reference (np.linalg.solve
 * always factorises, wmf_model.py:239); read after the stream has drained. */
int wmf_als_half_step_used_fallback(const void* ws, int* any_row_host, void* stream);

/* K3. Fused prediction + error reduction over the non-zero stored entries of a CSR matrix:
 * replaces predict + eval_prec (wmf_model.py:205-211, base_model.py:163-176).
 * Each prediction is computed in NumPy's rounding order (products rounded, pairwise reduce,
 * then + user bias + item bias). out[0] = sum (r-yhat)^2, out[1] = sum |r-yhat|, out[2] = count
 * (doubles; entries whose stored value is 0 are skipped like nonzero() does). Deterministic. */
size_t wmf_sddmm_loss_workspace_bytes(int64_t nnz);
int wmf_sddmm_loss(const int64_t* indptr, const int32_t* indices, const float* data, int64_t rows,
                   int64_t nnz, const float* U, int64_t ldu, const float* V, int64_t ldv, int f, int bias,
                   double* out3, void* ws, size_t ws_bytes, void* stream);

/* R8. Element-wise pair scores, bit-exact with NumPy:    replaces WMF.predict (:191-211).
 * users/items are int64 index arrays of length n; user_stride 0 broadcasts a single user. */
int wmf_predict_pairs(const int64_t* users, int64_t user_stride, const int64_t* items, int64_t n,
                      const float* U, int64_t ldu, const float* V, int64_t ldv, int f, int bias,
                      float* out, void* stream);

/* N2. Counting step of the sampled Recall@N protocol:    replaces the rank + `item in top[:k]` loop of
 * RecModel.compute_hit (base_model.py:84-95) for every held-out interaction at once.
 * S [nu x L] are the bit-exact scores (wmf_predict_pairs) of each user's drawn candidate list cand [nu x L]
 * (int32 item ids), slot[u] the position the held-out item overwrites (base_model.py:79-80). For interaction p
 * = (pair_user[p] = row of S/cand, pair_item[p], pair_score[p] = its exact score) ahead[p] receives the number
 * of candidates WMF.rank puts ahead of the item (higher score, or equal score at a lower position; a second
 * copy of the item id in the list counts as the item). The item is in top[:k] iff ahead[p] < k. */
int wmf_rank_ahead(const float* S, const int32_t* cand, const int32_t* slot, int64_t nu, int64_t L,
                   const int32_t* pair_user, const int32_t* pair_item, const float* pair_score, int64_t np,
                   int32_t* ahead, void* stream);

/* N5. Full-ranking quality of top-N lists (WMF.eval_ranking). No reference call site: the reference's only ranking
 * measure is the sampled Recall@N of eval_topn (N2 above). ids [nu x K] are the lists wmf_score_topk_exclude returns
 * (-1 padding is never a hit) for the users users[nu]; the test matrix t_* is a CSR indexed by user id with ids sorted
 * within each row, duplicates and explicit zeros allowed. T_u = the distinct ids of row u with a non-zero stored
 * value, h_i = hits among positions 1..i. For each cutoff k of ks_host (int32[nk], nk <= 16 distinct values in
 * [1, K]) per_user[(row * nk + j) * 5 + m] receives, for k = ks_host[j], m = 0..4:
 *   Recall h_k/|T_u|, Precision h_k/k, NDCG (sum of 1/log2(i+1) over hits i <= k) / (the same over i <= min(k,|T_u|)),
 *   MAP (sum of h_i/i over hits i <= k) / min(k,|T_u|), HitRate [h_k > 0],
 * or NaN for all of them when T_u is empty. Doubles, each user's row summed in an order fixed by its data alone.
 * wmf_topn_metrics_reduce: sums[nk*5 + 1] = the per-value sums over the rows whose first value is not NaN, then the
 * number of such rows; rows added in blocks whose size is fixed, the blocks in order (bitwise reproducible, whatever
 * calls filled per_user). */
size_t wmf_topn_metrics_workspace_bytes(int64_t nu, int nk);
int wmf_topn_metrics(const int64_t* ids, int64_t nu, int K, const int64_t* users, const int64_t* t_indptr,
                     const int32_t* t_indices, const float* t_data, const int32_t* ks_host, int nk, double* per_user,
                     void* stream);
int wmf_topn_metrics_reduce(const double* per_user, int64_t nu, int nk, double* sums, void* ws, size_t ws_bytes,
                            void* stream);

/* K4+K5. Top-N over a candidate list for a batch of users: replaces WMF.rank (:25-47).
 * Scores are the bit-exact fp32 scores of wmf_predict_pairs, so the selected index SET equals
 * the reference's; order is descending score, ties broken by lower candidate position.
 * When f (+1 with bias) <= 128, ni >= 256 and topn <= min(512, ni/32) the candidates come from a
 * tcgen05 FP16 GEMM with a proven error band and only they are rescored exactly (same lists as the
 * all-exact path, which the environment variable WMF_SCORE_EXACT=1 forces).
 * cand (nullable) = int64 candidate item ids [ni] (null: items 0..ni-1). out_ids [nu*topn]
 * receives item ids, out_scores (nullable) their scores. */
size_t wmf_score_topk_workspace_bytes(int64_t nu, int64_t ni, int topn);
int wmf_score_topk(const int64_t* users, int64_t nu, const int64_t* cand, int64_t ni, const float* U,
                   int64_t ldu, const float* V, int64_t ldv, int f, int bias, int topn, int64_t* out_ids,
                   float* out_scores, void* ws, size_t ws_bytes, void* stream);
/* K4+K5 with exclusion: top-N over all items 0..ni-1 minus the items each user has interacted with: replaces the
 * rank(np.delete(all_items, seen)) loop of test_coverage (RecModel/utils.py:3-18).
 * ex_indptr int64[rows+1] / ex_indices int32 are a CSR matrix whose row `user` lists the item ids to leave out for
 * that user (rows indexed by user id, ids in [0, ni) sorted ascending within each row, duplicates allowed; values
 * are not read). Same scores, order and tie rule as wmf_score_topk over the remaining items; a user with fewer than
 * topn of them gets id -1 (score NaN) in the rest of its row. The tensor-core path masks the excluded ids in both
 * GEMM passes; a user whose candidate list overflows makes the exact kernels redo the call, and fixup_users
 * (nullable, device int32) receives the number of such users (0: the tensor-core path alone answered). */
size_t wmf_score_topk_exclude_workspace_bytes(int64_t nu, int64_t ni, int topn);
int wmf_score_topk_exclude(const int64_t* users, int64_t nu, const int64_t* ex_indptr, const int32_t* ex_indices,
                           int64_t ni, const float* U, int64_t ldu, const float* V, int64_t ldv, int f, int bias,
                           int topn, int64_t* out_ids, float* out_scores, int32_t* fixup_users, void* ws,
                           size_t ws_bytes, void* stream);

/* K7. Unweighted half-step X = R * (Ginv * Y^T)^T:       replaces wmf_model.py:85,:88.
 * wmf_inverse: Ginv = inv(G) for a small dense f x f matrix (np.linalg.inv), one CTA.
 * wmf_dense_right_multiply: W[n x f] = Y[n x f] * M[f x f]^T   (= (M Y^T)^T).
 * wmf_spmm: X[r] = sum_j data_j * W[indices_j]                 (csr_matrix.dot). */
int wmf_inverse(const float* G, int f, float* Ginv, void* ws, size_t ws_bytes, void* stream);
size_t wmf_inverse_workspace_bytes(int f);
int wmf_dense_right_multiply(const float* Y, int64_t n, int64_t ldy, const float* M, int f, float* W,
                             int64_t ldw, void* stream);
int wmf_spmm(const int64_t* indptr, const int32_t* indices, const float* data, int64_t rows,
             const float* W, int64_t ldw, int f, float* X, int64_t ldx, void* stream);

/* N4. EASE, the WMF path's dense sibling:                replaces Ease.train (RecModel/ease_model.py:81-114) and
 * _predict_ease (RecModel/fast_utils/ease_utils.pyx:15-30).
 * wmf_ease_train: W[n x n] (row-major, ld = n) = P / (-diag(P) + 1e-9) column-wise with a zero diagonal, where
 * P = inv(X^T X + alpha I) and X is the `rows` x n interaction matrix in CSR (Gram by one warp per user row, blocked
 * in-place Gauss-Jordan inverse in FP32: G is symmetric positive definite, no pivoting).
 * wmf_ease_predict: out[k] = sum_j X[users[k*user_stride], j] * W[j, items[k]] with FP32 products summed in double in
 * stored order (what the reference's Cython loop does); user_stride 0 broadcasts one user. */
size_t wmf_ease_workspace_bytes(int64_t n);
int wmf_ease_train(const int64_t* indptr, const int32_t* indices, const float* data, int64_t rows, int64_t n, float alpha,
                   float* W, void* ws, size_t ws_bytes, void* stream);
int wmf_ease_predict(const int64_t* indptr, const int32_t* indices, const float* data, const float* W, int64_t n,
                     const int64_t* users, int64_t user_stride, const int64_t* items, int64_t count, double* out,
                     void* stream);
/* N4 ranking: top-N of all n items minus the ones each user has interacted with, for nu users in one call: replaces
 * the per-user Ease.rank(np.delete(all_items, seen), user) loop of test_coverage (RecModel/utils.py:3-18). No
 * reference call site ranks EASE over all items in one call.
 * Score s(u, i) = the sum over the stored entries e of row u of X (x_*, in stored order, from +0.0) of
 * (double)(x_e * W[j_e, i]) with the product rounded to FP32: bitwise what wmf_ease_predict returns. Unsorted rows,
 * duplicates and explicit zeros in X take part as stored. The double scores are ranked as they are (no FP32 rounding),
 * descending, ties to the lower item id. ex_indptr (nullable: nothing excluded) / ex_indices: a CSR indexed by user
 * id whose row users[k] lists the item ids to leave out (unsorted rows and duplicates allowed, values not read).
 * out_ids [nu*topn] receives item ids, out_scores (nullable) [nu*topn] their scores; a user with fewer than topn
 * unseen items gets id -1 and score NaN in the rest of its row. 1 <= topn <= min(n, 1024) (else
 * WMF_ERR_UNSUPPORTED), 0 < n < 2^31. The workspace holds one [ub x n] double score tile, ub from n and a fixed
 * byte budget. */
size_t wmf_ease_score_topk_workspace_bytes(int64_t nu, int64_t n, int topn);
int wmf_ease_score_topk(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data, const float* W,
                        int64_t n, const int64_t* users, int64_t nu, const int64_t* ex_indptr,
                        const int32_t* ex_indices, int topn, int64_t* out_ids, double* out_scores, void* ws,
                        size_t ws_bytes, void* stream);

/* ItemKNN: an item-item neighbourhood model (DESIGN.md 4.6). No reference call site: the neighbourhood sources of
 * RecModel are not part of this repository, and this model is defined here, not ported.
 * X is the `rows` x n interaction matrix in canonical CSR: sorted column indices, no duplicates, no explicit zeros
 * (duplicates would count twice; scores walk each row in stored order). P is its binary pattern and
 * c_ab = sum_u P[u, a] P[u, b], an exact integer; c_aa is the number of users of a.
 * wmf_knn_train: sim(a, b) in double, every operation rounded to nearest, no fused multiply-add:
 *   WMF_KNN_COSINE       c_ab / (sqrt(c_aa) * sqrt(c_bb) + shrink)
 *   WMF_KNN_JACCARD      c_ab / ((c_aa + c_bb - c_ab) + shrink)
 *   WMF_KNN_CONDITIONAL  c_ab / (c_aa + shrink)            (P(b | a): W is not symmetric)
 * Row a of W holds the top-min(k, n) items b != a with c_ab > 0 by sim(a, b), ties to the lower id, fewer when a has
 * fewer such items; W[a, b] = sim(a, b). W is written as an n x n CSR with sorted column indices: w_indptr [n+1], and
 * w_indices / w_data with room for n * min(k, n) entries, of which the first w_indptr[n] are used. xt_indptr /
 * xt_indices: the CSR of X^T (wmf_csr_transpose). 1 <= k <= 1024, similarity one of WMF_KNN_*, shrink finite and
 * >= 0, 0 < n < 2^31: else WMF_ERR_INVALID before any CUDA call. The workspace holds an int32 and a double [B x n]
 * tile (B item rows from n and a fixed byte budget) and the selected rows of all n items. Called with the roles of X
 * and X^T swapped (x_* = the CSR of X^T, rows = the item count, xt_* = the CSR of X, n = the user count), it writes
 * the user-user neighbours of UserKNN: c_ab is then the number of items users a and b share.
 * wmf_knn_predict: out[k] = s(users[k*user_stride], items[k]); user_stride 0 broadcasts one user. The score
 * s(u, i) is the sum over the entries j of row u of X, in ascending j, from +0.0, of (double)x_uj * W[j, i], each
 * product and each addition rounded to nearest; an item no entry of W votes for scores +0.0. W is any n x n CSR
 * with sorted column indices (w_data double).
 * wmf_knn_score_topk: wmf_ease_score_topk's contract (exclusion CSR, ordering, -1 / NaN padding, 1 <= topn <=
 * min(n, 1024) else WMF_ERR_UNSUPPORTED) with the scores of wmf_knn_predict, bitwise. The workspace holds one
 * [ub x n] double score tile. */
#define WMF_KNN_COSINE 0
#define WMF_KNN_JACCARD 1
#define WMF_KNN_CONDITIONAL 2
size_t wmf_knn_train_workspace_bytes(int64_t n, int k);
int wmf_knn_train(const int64_t* x_indptr, const int32_t* x_indices, int64_t rows, const int64_t* xt_indptr,
                  const int32_t* xt_indices, int64_t n, int k, int similarity, double shrink, int64_t* w_indptr,
                  int32_t* w_indices, double* w_data, void* ws, size_t ws_bytes, void* stream);
int wmf_knn_predict(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data, const int64_t* w_indptr,
                    const int32_t* w_indices, const double* w_data, const int64_t* users, int64_t user_stride,
                    const int64_t* items, int64_t count, double* out, void* stream);
size_t wmf_knn_score_topk_workspace_bytes(int64_t nu, int64_t n, int topn);
int wmf_knn_score_topk(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data, const int64_t* w_indptr,
                       const int32_t* w_indices, const double* w_data, int64_t n, const int64_t* users, int64_t nu,
                       const int64_t* ex_indptr, const int32_t* ex_indices, int topn, int64_t* out_ids,
                       double* out_scores, void* ws, size_t ws_bytes, void* stream);

/* UserKNN: a user-user neighbourhood model (DESIGN.md 4.8), defined here, not ported. X is the canonical interaction
 * matrix of the knn entries above (users x n items; sorted rows, no duplicates, no explicit zeros: not checked, a
 * duplicate item in a row would race in the score tile). nb_indptr / nb_indices / nb_data: the neighbour CSR N, one
 * row per user of X with sorted column indices (user ids) and double similarities, as wmf_knn_train writes it for
 * (X^T, X).
 * wmf_userknn_predict: out[k] = s(users[k*user_stride], items[k]); user_stride 0 broadcasts one user. The score
 * s(u, i) is the sum over the entries v of row u of N, in ascending v, from +0.0, of sim(u, v) * (double)x_vi, each
 * product and each addition rounded to nearest; an item no neighbour of u has scores +0.0. count < 0 or
 * user_stride < 0: WMF_ERR_INVALID, count 0: WMF_OK with nothing read; a null pointer otherwise: WMF_ERR_INVALID.
 * All before any CUDA call.
 * wmf_userknn_score_topk: wmf_knn_score_topk's contract (exclusion CSR by user id, descending scores, ties to the
 * lower item id, -1 / NaN padding, 1 <= topn <= min(n, 1024) else WMF_ERR_UNSUPPORTED, the same order of checks)
 * with the scores of wmf_userknn_predict, bitwise. n is the item count. The workspace
 * (wmf_userknn_score_topk_workspace_bytes, 0 for nu <= 0 or n outside 1..2^31-1) holds one [ub x n] double score
 * tile, ub from n and a fixed byte budget. */
int wmf_userknn_predict(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data,
                        const int64_t* nb_indptr, const int32_t* nb_indices, const double* nb_data,
                        const int64_t* users, int64_t user_stride, const int64_t* items, int64_t count, double* out,
                        void* stream);
size_t wmf_userknn_score_topk_workspace_bytes(int64_t nu, int64_t n, int topn);
int wmf_userknn_score_topk(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data,
                           const int64_t* nb_indptr, const int32_t* nb_indices, const double* nb_data, int64_t n,
                           const int64_t* users, int64_t nu, const int64_t* ex_indptr, const int32_t* ex_indices,
                           int topn, int64_t* out_ids, double* out_scores, void* ws, size_t ws_bytes, void* stream);

/* UserKNN fold-in (DESIGN.md 4.10): the neighbours among the m training users of nq new histories that are not rows
 * of X. q_indptr / q_indices: the new rows, canonical like X (sorted, no duplicates, no explicit zeros: not checked,
 * a duplicate would count twice), column ids below n_items. xt_indptr / xt_indices: the CSR of the training X^T
 * (n_items rows, each item's users); x_indptr: the m + 1 row offsets of the training X. With q_r the pattern of new
 * row r and P_v that of training user v, c_rv = |q_r ∩ P_v|, c_rr = |q_r| and c_vv = |P_v| (exact integers), and
 * sim(r, v) is wmf_knn_train's formula for `similarity` and `shrink`. Row r of the output N' holds the top-min(k, m)
 * training users v with c_rv > 0 by sim(r, v), ties to the lower id (no self exclusion: r is not a training user);
 * N'[r, v] = sim(r, v). N' is written as an nq x m CSR with sorted column indices (out_indptr [nq+1], out_indices /
 * out_data with room for nq * min(k, m) entries, the first out_indptr[nq] used): the layout wmf_userknn_predict and
 * wmf_userknn_score_topk take, indexed by new-row id. 1 <= k <= 1024, similarity one of WMF_KNN_*, shrink finite and
 * >= 0, 0 < m < 2^31, 0 < nq < 2^31, n_items >= 0, non-null pointers (q_indices / xt_indices may be null when they
 * hold no entry): else WMF_ERR_INVALID before any CUDA call; a short workspace: WMF_ERR_WORKSPACE. The workspace
 * (wmf_userknn_fold_in_workspace_bytes, 0 for arguments out of range) holds an int32 and a double [B x m] tile (B new
 * rows from m and a fixed byte budget) and the selected rows of all nq histories. */
size_t wmf_userknn_fold_in_workspace_bytes(int64_t nq, int64_t m, int k);
int wmf_userknn_fold_in(const int64_t* q_indptr, const int32_t* q_indices, int64_t nq, const int64_t* xt_indptr,
                        const int32_t* xt_indices, int64_t n_items, const int64_t* x_indptr, int64_t m, int k,
                        int similarity, double shrink, int64_t* out_indptr, int32_t* out_indices, double* out_data,
                        void* ws, size_t ws_bytes, void* stream);

/* SLIM: sparse non-negative item-item regression (DESIGN.md 4.7). No reference call site: the SLIM sources of
 * RecModel are not part of this repository, and this model is defined here, not ported.
 * X, X^T and P are those of the knn entries above (canonical X); G = P^T P, so G[a, b] = c_ab. The candidates S_j of
 * item j are row j of cand_indptr / cand_indices (wmf_knn_train's W with WMF_KNN_COSINE and shrink 0 is the intended
 * source). Each row must be ascending, hold no self entry (j itself) and be no longer than k: not checked. Column j
 * of W solves  min_w 1/2 |P[:, j] - P[:, S_j] w|^2 + l1 sum(w) + l2/2 |w|^2,  w >= 0, by cyclic coordinate descent on
 * G_S = G[S_j, S_j] and b = G[S_j, j] in double, every operation rounded to nearest, none fused:
 *   w = 0, q = b; per sweep: d = wm = 0; for p in order: z = q[p] + G_S[p,p] w[p];
 *   new = z > l1 ? (z - l1) / (G_S[p,p] + l2) : 0; if new != w[p]: q[r] -= G_S[r,p] (new - w[p]) for all r, w[p] = new;
 *   d = max(d, |new - old|), wm = max(wm, |new|); stop when wm == 0, d <= tol wm, or after max_iter sweeps.
 * W^T is written as an n x n CSR (row j = column j of W: the candidates with w > 0, ascending ids): wt_indptr [n+1],
 * and wt_indices / wt_data with room for n * min(k, n) entries, of which the first wt_indptr[n] are used.
 * sweeps [n] (int32) receives the number of sweeps run per column. 1 <= k <= 128, l1 and l2 finite and >= 0,
 * max_iter >= 1, tol finite and >= 0, 0 < n <= 2^30: else WMF_ERR_INVALID before any CUDA call. The workspace holds
 * the dense int32 G (n^2 * 4 bytes, 64-bit offsets) and the staged columns. */
size_t wmf_slim_train_workspace_bytes(int64_t n, int k);
int wmf_slim_train(const int64_t* x_indptr, const int32_t* x_indices, int64_t rows, const int64_t* xt_indptr,
                   const int32_t* xt_indices, int64_t n, const int64_t* cand_indptr, const int32_t* cand_indices, int k,
                   double l1, double l2, int max_iter, double tol, int64_t* wt_indptr, int32_t* wt_indices,
                   double* wt_data, int32_t* sweeps, void* ws, size_t ws_bytes, void* stream);

/* RP3beta: a three-step random walk user -> item -> user -> item in closed form (DESIGN.md 4.9), defined here, not
 * ported. P (p_indptr / p_indices, `rows` x n) is the binary pattern of the canonical X of the knn entries above (sorted
 * rows, no duplicates: not checked, a duplicate item in a row would race in the tile); pt_* is the CSR of P^T
 * (wmf_csr_transpose: each item's users ascending); nnz = p_indptr[rows] = pt_indptr[n]. du [rows], ra [n], cb [n] are
 * the caller's scales (deg_u^-alpha, pop_a^-alpha, pop_b^-beta, computed on the host; entries of empty rows and
 * columns are not read); no device code calls pow. In double, every operation rounded to nearest, none fused:
 *   S_ab = sum over the users u of both a and b, ascending, from +0.0, of du[u];   W'_ab = (ra[a] * S_ab) * cb[b].
 * Row a of W holds the top-min(k, n) items b != a with S_ab > 0 by W'_ab, ties to the lower id, fewer when a has fewer
 * such items; W[a, b] = W'_ab, written like wmf_knn_train's W (n x n CSR, sorted rows, room for n * min(k, n)
 * entries, the first w_indptr[n] used), so wmf_knn_predict and wmf_knn_score_topk score it. 1 <= k <= 1024,
 * 0 < n < 2^31, rows >= 0, 0 <= nnz < 2^40, non-null pointers (p_indices / pt_indices may be null when nnz is 0, du
 * when rows is 0): else WMF_ERR_INVALID before any CUDA call; a short workspace: WMF_ERR_WORKSPACE. The workspace
 * (wmf_rp3beta_train_workspace_bytes, 0 for arguments out of range) holds a double [B x n] tile (B item rows from n
 * and a fixed byte budget), the selected rows of all n items, the item order and nnz walk weights. */
size_t wmf_rp3beta_train_workspace_bytes(int64_t n, int64_t nnz, int k);
int wmf_rp3beta_train(const int64_t* p_indptr, const int32_t* p_indices, int64_t rows, const int64_t* pt_indptr,
                      const int32_t* pt_indices, int64_t n, int64_t nnz, const double* du, const double* ra,
                      const double* cb, int k, int64_t* w_indptr, int32_t* w_indices, double* w_data, void* ws,
                      size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* WMF_B200_H */
