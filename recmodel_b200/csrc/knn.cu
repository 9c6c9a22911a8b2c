// ItemKNN: an item-item neighbourhood model (DESIGN.md 4.6). For the users x n binary pattern P of the canonical X:
//   c_ab = sum_u P[u, a] P[u, b]                          -> knn_cooc_kernel (int32 counts, [B x n] tile per item block)
//   sim(a, b) from c_ab, c_aa, c_bb, shrink                -> knn_similarity_kernel (double, no FMA contraction)
//   W[a, :] = top-k of sim(a, b), b != a, c_ab > 0          -> topk_rows_kernel<double> (score.cu), knn_sort_rows_kernel
//   s(u, i) = sum over j of row u, ascending, of x_uj W[j, i] -> knn_score_tile_kernel (recommend), knn_predict_kernel
// Every double operation is an explicit round-to-nearest intrinsic, so a NumPy restatement of the definitions
// reproduces each similarity and each score bitwise.
// SLIM (DESIGN.md 4.7) shares the counts, the staging-to-CSR kernels and the scoring: the dense G = P^T P comes from
// knn_cooc_kernel over all n rows, slim_cd_kernel solves each column's regression on chip, and knn_scan_kernel plus
// knn_compact_kernel write the CSR of W^T.
// UserKNN (DESIGN.md 4.8) trains with wmf_knn_train on (X^T, X) and scores with userknn_score_tile_kernel and
// userknn_predict_kernel, which walk the neighbours' rows of X. Its fold-in (DESIGN.md 4.10, wmf_userknn_fold_in)
// counts new rows against the training users with knn_cooc_kernel, scores them with
// userknn_cross_similarity_kernel and selects and writes the neighbours like wmf_knn_train.
// RP3beta (DESIGN.md 4.9) sums its walk weights into a [B x n] tile with userknn_score_tile_kernel over (P^T, P), rows
// grouped by walk length (rp3_chain_kernel, rp3_order_kernel), scales them (rp3_weight_kernel), selects like ItemKNN
// and sorts each row into the staging row of its item (rp3_sort_rows_kernel); W is then scored like ItemKNN's.
#include "common.cuh"
#include "score.cuh"

namespace wmf {

namespace {

constexpr int KN_THREADS = 256;
constexpr size_t KN_TILE_BYTES = 64ull << 20;   // double tiles near 64 MiB: the selection passes stay in L2 (126 MB)

__device__ __forceinline__ double knn_pop(const int64_t* __restrict__ xt_indptr, int64_t a) {
    return (double)(xt_indptr[a + 1] - xt_indptr[a]);
}

// C[a - a0][j] += 1 for every stored entry (a, u) of rows [a0, a0 + B) of X^T and every stored entry j of row u of X.
// One warp per (a, u) entry, flattened over the block so that a popular item spreads over many warps; lanes over row
// u. The integer atomics make the counts independent of the order.
__global__ __launch_bounds__(KN_THREADS) void knn_cooc_kernel(const int64_t* __restrict__ x_indptr,
                                                              const int32_t* __restrict__ x_indices,
                                                              const int64_t* __restrict__ xt_indptr,
                                                              const int32_t* __restrict__ xt_indices, int64_t n,
                                                              int64_t a0, int B, int* __restrict__ C) {
    const int64_t base = xt_indptr[a0], cnt = xt_indptr[a0 + B] - base;
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < cnt; w += warps) {
        const int64_t e = base + w;
        int lo = 0, hi = B - 1;   // the block row holding entry e: the last r with xt_indptr[a0 + r] <= e
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (xt_indptr[a0 + mid] <= e) lo = mid; else hi = mid - 1;
        }
        const int64_t u = xt_indices[e];
        int* crow = C + (int64_t)lo * n;
        for (int64_t t = x_indptr[u] + lane; t < x_indptr[u + 1]; t += 32) atomicAdd(crow + x_indices[t], 1);
    }
}

// sim(a, b) from c_ab, c_aa and c_bb: the formulas of wmf_knn_train, every operation rounded to nearest, none fused
__device__ __forceinline__ double knn_sim(int sim, double cab, double caa, double cbb, double shrink) {
    double den;
    if (sim == WMF_KNN_COSINE) den = __dadd_rn(__dmul_rn(__dsqrt_rn(caa), __dsqrt_rn(cbb)), shrink);
    else if (sim == WMF_KNN_JACCARD) den = __dadd_rn(__dsub_rn(__dadd_rn(caa, cbb), cab), shrink);
    else den = __dadd_rn(caa, shrink);
    return __ddiv_rn(cab, den);
}

// S[r][b] = sim(a0 + r, b) from the counts; self and c_ab = 0 get RankKey<double>::excluded(). c_bb is the column
// count of X (X^T row length): the canonical X stores each (u, b) once.
__global__ __launch_bounds__(KN_THREADS) void knn_similarity_kernel(const int* __restrict__ C,
                                                                    const int64_t* __restrict__ xt_indptr, int64_t n,
                                                                    int64_t a0, int sim, double shrink,
                                                                    double* __restrict__ S) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const int64_t r = blockIdx.y, a = a0 + r, e = r * n + b;
    const int c = C[e];
    double s = RankKey<double>::excluded();
    if (c != 0 && b != a) s = knn_sim(sim, (double)c, knn_pop(xt_indptr, a), knn_pop(xt_indptr, b), shrink);
    S[e] = s;
}

// The body of the row sorts below, for one CTA: the selected (id, value) pairs of selection row r (ids -1 where the
// row had fewer than kk candidates) sorted by id into row `row` of the [n x kk] staging area; cnt[row] = their number.
// The rank of an entry is the number of selected ids below it (ids are distinct).
__device__ __forceinline__ void knn_sort_row(const int64_t* __restrict__ ids, const double* __restrict__ vals, int kk,
                                             int64_t r, int64_t row, int32_t* __restrict__ st_idx,
                                             double* __restrict__ st_val, int64_t* __restrict__ cnt) {
    __shared__ int32_t sid[TK_MAX];
    __shared__ unsigned s_m;
    if (threadIdx.x == 0) s_m = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < kk; t += KN_THREADS) {
        const int32_t id = (int32_t)ids[r * kk + t];
        sid[t] = id;
        if (id >= 0) atomicAdd(&s_m, 1u);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < kk; t += KN_THREADS) {
        const int32_t id = sid[t];
        if (id < 0) continue;
        int pos = 0;
        for (int q = 0; q < kk; ++q) pos += (sid[q] >= 0 && sid[q] < id);
        st_idx[row * kk + pos] = id;
        st_val[row * kk + pos] = vals[r * kk + t];
    }
    if (threadIdx.x == 0) cnt[row] = s_m;
}

// One CTA per block row: selection row r into staging row a0 + r
__global__ __launch_bounds__(KN_THREADS) void knn_sort_rows_kernel(const int64_t* __restrict__ ids,
                                                                   const double* __restrict__ vals, int kk, int64_t a0,
                                                                   int32_t* __restrict__ st_idx,
                                                                   double* __restrict__ st_val,
                                                                   int64_t* __restrict__ cnt) {
    knn_sort_row(ids, vals, kk, blockIdx.x, a0 + blockIdx.x, st_idx, st_val, cnt);
}

// indptr[0] = 0, indptr[a + 1] = cnt[0] + ... + cnt[a]: one CTA, chunks of KN_THREADS rows
__global__ __launch_bounds__(KN_THREADS) void knn_scan_kernel(const int64_t* __restrict__ cnt, int64_t n,
                                                              int64_t* __restrict__ indptr) {
    __shared__ int64_t warp_tot[KN_THREADS / 32];
    __shared__ int64_t s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { s_carry = 0; indptr[0] = 0; }
    __syncthreads();
    for (int64_t c0 = 0; c0 < n; c0 += KN_THREADS) {
        const int64_t a = c0 + tid;
        int64_t v = a < n ? cnt[a] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += y;
        }
        if (lane == 31) warp_tot[warp] = v;
        __syncthreads();
        int64_t before = s_carry;
        for (int w = 0; w < warp; ++w) before += warp_tot[w];
        if (a < n) indptr[a + 1] = before + v;
        __syncthreads();
        if (tid == KN_THREADS - 1) s_carry = before + v;
        __syncthreads();
    }
}

// the staged rows into the CSR: one warp per row
__global__ __launch_bounds__(KN_THREADS) void knn_compact_kernel(const int32_t* __restrict__ st_idx,
                                                                 const double* __restrict__ st_val, int kk, int64_t n,
                                                                 const int64_t* __restrict__ indptr,
                                                                 int32_t* __restrict__ w_indices,
                                                                 double* __restrict__ w_data) {
    const int64_t a = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (a >= n) return;
    const int lane = threadIdx.x & 31;
    const int64_t lo = indptr[a], m = indptr[a + 1] - lo;
    for (int64_t t = lane; t < m; t += 32) {
        w_indices[lo + t] = st_idx[a * kk + t];
        w_data[lo + t] = st_val[a * kk + t];
    }
}

// S[r][i] = s(users[u_begin + r], i) on a zeroed [ub x n] tile. One warp per user walks row u of X in ascending j
// (32 entries and their W row bounds fetched at once, then broadcast); lanes over the entries of W row j, which are
// distinct ids. The __syncwarp between rows j orders the read-modify-writes of one item, so every score is summed
// from +0.0 in ascending j without atomics: the sum of knn_predict_kernel.
__global__ __launch_bounds__(KN_THREADS) void knn_score_tile_kernel(
    const int64_t* __restrict__ x_indptr, const int32_t* __restrict__ x_indices, const float* __restrict__ x_data,
    const int64_t* __restrict__ w_indptr, const int32_t* __restrict__ w_indices, const double* __restrict__ w_data,
    int64_t n, const int64_t* __restrict__ users, int64_t u_begin, int ub, double* S) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= ub) return;
    const int lane = threadIdx.x & 31;
    const int64_t u = users[u_begin + r];
    const int64_t hi = x_indptr[u + 1];
    double* srow = S + r * n;
    for (int64_t e0 = x_indptr[u]; e0 < hi; e0 += 32) {
        double x = 0.0;
        int64_t wlo = 0, whi = 0;
        if (e0 + lane < hi) {
            const int32_t j = x_indices[e0 + lane];
            x = (double)x_data[e0 + lane];
            wlo = w_indptr[j];
            whi = w_indptr[j + 1];
        }
        const int m = (int)(hi - e0 < 32 ? hi - e0 : 32);
        for (int q = 0; q < m; ++q) {
            const double xq = __shfl_sync(0xffffffffu, x, q);
            const int64_t lo = __shfl_sync(0xffffffffu, wlo, q), end = __shfl_sync(0xffffffffu, whi, q);
            for (int64_t t = lo + lane; t < end; t += 32) {
                const int32_t i = w_indices[t];
                srow[i] = __dadd_rn(srow[i], __dmul_rn(xq, w_data[t]));
            }
            __syncwarp();
        }
    }
}

// out[k] = s(users[k * user_stride], items[k]): row u of X in ascending j, a binary search of the item in W row j
__global__ __launch_bounds__(KN_THREADS) void knn_predict_kernel(
    const int64_t* __restrict__ x_indptr, const int32_t* __restrict__ x_indices, const float* __restrict__ x_data,
    const int64_t* __restrict__ w_indptr, const int32_t* __restrict__ w_indices, const double* __restrict__ w_data,
    const int64_t* __restrict__ users, int64_t user_stride, const int64_t* __restrict__ items, int64_t count,
    double* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const int64_t u = users[k * user_stride];
    const int32_t it = (int32_t)items[k];
    double acc = 0.0;
    for (int64_t e = x_indptr[u]; e < x_indptr[u + 1]; ++e) {
        const int32_t j = x_indices[e];
        int64_t lo = w_indptr[j], hi = w_indptr[j + 1];   // first entry >= it
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (w_indices[mid] < it) lo = mid + 1; else hi = mid;
        }
        if (lo < w_indptr[j + 1] && w_indices[lo] == it) acc = __dadd_rn(acc, __dmul_rn((double)x_data[e], w_data[lo]));
    }
    out[k] = acc;
}

// ---- UserKNN (DESIGN.md 4.8): the neighbour CSR N (n_users x n_users) is wmf_knn_train's W for (X^T, X), and a
// user's neighbours vote through their rows of X: s(u, i) = sum over v of row u of N, ascending, of sim(u, v) x_vi.

// S[r][i] = s(users[u_begin + r], i) on a zeroed [ub x n] tile. One CTA per user: the neighbours v of row u of N are
// staged KN_THREADS at a time (X row bounds, similarity) in shared memory, then walked in ascending v with the
// threads over the entries of X row v, which are distinct items. X rows are long-tailed (thousands of entries), so a
// whole CTA walks each one. The __syncthreads between rows v orders the read-modify-writes of one item, so every
// score is summed from +0.0 in ascending v without atomics: the sum of userknn_predict_kernel.
__global__ __launch_bounds__(KN_THREADS) void userknn_score_tile_kernel(
    const int64_t* __restrict__ x_indptr, const int32_t* __restrict__ x_indices, const float* __restrict__ x_data,
    const int64_t* __restrict__ nb_indptr, const int32_t* __restrict__ nb_indices, const double* __restrict__ nb_data,
    int64_t n, const int64_t* __restrict__ users, int64_t u_begin, double* S) {
    __shared__ int64_t s_lo[KN_THREADS], s_hi[KN_THREADS];
    __shared__ double s_sim[KN_THREADS];
    const int64_t r = blockIdx.x;
    const int64_t u = users[u_begin + r];
    const int64_t hi = nb_indptr[u + 1];
    double* srow = S + r * n;
    for (int64_t e0 = nb_indptr[u]; e0 < hi; e0 += KN_THREADS) {
        const int m = (int)(hi - e0 < KN_THREADS ? hi - e0 : KN_THREADS);
        if ((int)threadIdx.x < m) {
            const int32_t v = nb_indices[e0 + threadIdx.x];
            s_lo[threadIdx.x] = x_indptr[v];
            s_hi[threadIdx.x] = x_indptr[v + 1];
            s_sim[threadIdx.x] = nb_data[e0 + threadIdx.x];
        }
        __syncthreads();
        for (int q = 0; q < m; ++q) {
            const double sim = s_sim[q];
            const int64_t end = s_hi[q];
            for (int64_t t = s_lo[q] + threadIdx.x; t < end; t += KN_THREADS) {
                const int32_t i = x_indices[t];
                srow[i] = __dadd_rn(srow[i], __dmul_rn(sim, (double)x_data[t]));
            }
            __syncthreads();   // also ends the reads of the staged chunk before the next one overwrites it
        }
    }
}

// out[k] = s(users[k * user_stride], items[k]): row u of N in ascending v, a binary search of the item in X row v
__global__ __launch_bounds__(KN_THREADS) void userknn_predict_kernel(
    const int64_t* __restrict__ x_indptr, const int32_t* __restrict__ x_indices, const float* __restrict__ x_data,
    const int64_t* __restrict__ nb_indptr, const int32_t* __restrict__ nb_indices, const double* __restrict__ nb_data,
    const int64_t* __restrict__ users, int64_t user_stride, const int64_t* __restrict__ items, int64_t count,
    double* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const int64_t u = users[k * user_stride];
    const int32_t it = (int32_t)items[k];
    double acc = 0.0;
    for (int64_t e = nb_indptr[u]; e < nb_indptr[u + 1]; ++e) {
        const int32_t v = nb_indices[e];
        int64_t lo = x_indptr[v], hi = x_indptr[v + 1];   // first entry >= it
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (x_indices[mid] < it) lo = mid + 1; else hi = mid;
        }
        if (lo < x_indptr[v + 1] && x_indices[lo] == it)
            acc = __dadd_rn(acc, __dmul_rn(nb_data[e], (double)x_data[lo]));
    }
    out[k] = acc;
}

// Fold-in (DESIGN.md 4.10): S[r][v] = sim(q_{r0 + r}, v) between new row r0 + r of Q and training user v from the
// counts C[r][v] = |q_r ∩ P_v|; c_rr is the Q row length, c_vv the X row length (both canonical). c_rv = 0 gets
// RankKey<double>::excluded(); there is no self to exclude, r is not a training user.
__global__ __launch_bounds__(KN_THREADS) void userknn_cross_similarity_kernel(const int* __restrict__ C,
                                                                              const int64_t* __restrict__ q_indptr,
                                                                              const int64_t* __restrict__ x_indptr,
                                                                              int64_t m, int64_t r0, int sim,
                                                                              double shrink, double* __restrict__ S) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= m) return;
    const int64_t r = blockIdx.y, e = r * m + v;
    const int c = C[e];
    S[e] = c != 0 ? knn_sim(sim, (double)c, knn_pop(q_indptr, r0 + r), knn_pop(x_indptr, v), shrink)
                  : RankKey<double>::excluded();
}

// rows per [B x n] similarity tile (and users per score tile): the double tile near KN_TILE_BYTES, at least one row
int64_t knn_batch(int64_t rows, int64_t n) {
    int64_t b = (int64_t)(KN_TILE_BYTES / ((size_t)n * 8));
    if (b < 1) b = 1;
    if (b > rows) b = rows;
    return b;
}

struct TrainLayout {
    size_t C, S, ids, vals, st_idx, st_val, cnt, total;
};

// rows per fold-in tile: knn_batch, at most 65535 (the similarity kernel's grid rows; training tiles stay below 2 897)
int64_t fold_in_batch(int64_t nq, int64_t m) {
    const int64_t b = knn_batch(nq, m);
    return b < 65535 ? b : 65535;
}

// `rows` selection rows over n columns in tiles of B rows: wmf_knn_train has rows = n, the fold-in one row per history
TrainLayout train_layout(int64_t rows, int64_t n, int kk, size_t B) {
    TrainLayout L;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t at = off; off += align_up(bytes, 256); return at; };
    L.C = take(B * n * 4);
    L.S = take(B * n * 8);
    L.ids = take(B * kk * 8);
    L.vals = take(B * kk * 8);
    L.st_idx = take((size_t)rows * kk * 4);
    L.st_val = take((size_t)rows * kk * 8);
    L.cnt = take((size_t)rows * 8);
    L.total = off;
    return L;
}

// ---- SLIM (DESIGN.md 4.7): one non-negative elastic-net regression per item column over its candidates, by cyclic
// coordinate descent on the Gram G = P^T P, whose dense n x n int32 form knn_cooc_kernel writes (a0 = 0, B = n).

constexpr int SL_MAX = 128;   // largest candidate list: the int32 G_S of 128 x 128 is 64 KB of shared memory

__device__ __forceinline__ double sl_pick(const double (&v)[4], int t) {
    return t == 0 ? v[0] : t == 1 ? v[1] : t == 2 ? v[2] : v[3];
}

// the first set bit at or after `from` in the 128-bit mask act, SL_MAX when there is none
__device__ __forceinline__ int sl_next(const unsigned (&act)[4], int from) {
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int lo = from - 32 * t;
        unsigned mk = lo >= 32 ? 0u : act[t];
        if (lo > 0 && lo < 32) mk &= ~0u << lo;
        if (mk) return 32 * t + __ffs(mk) - 1;
    }
    return SL_MAX;
}

// One warp per item column j. Lane l owns coordinates r = l + 32 t (t < 4): the candidate id s_r, q[r] and w[r] in
// registers. G_S = G[S_j, S_j] (int32, row p at Gs + p m) stays in shared memory for the whole solve; G is symmetric,
// so the column G_S[:, p] an update reads is row p, one conflict-free word per lane. Every lane runs the scalar part
// of each step (same values), so the loop bounds, d and wm are warp-uniform. A ballot marks the coordinates that can
// change (w != 0 or q > l1); the others are skipped, which changes no bit of the defined loop. The positive w go to
// row j of the [n x kk] staging area in ascending id order, their number to cnt[j].
__global__ __launch_bounds__(32) void slim_cd_kernel(const int* __restrict__ G, int64_t n,
                                                     const int64_t* __restrict__ cand_indptr,
                                                     const int32_t* __restrict__ cand_indices, int kk, double l1,
                                                     double l2, int max_iter, double tol, int32_t* __restrict__ st_idx,
                                                     double* __restrict__ st_val, int64_t* __restrict__ cnt,
                                                     int32_t* __restrict__ sweeps) {
    extern __shared__ int sl_smem[];
    int* Gs = sl_smem;
    int* ids = sl_smem + (size_t)kk * kk;
    const int64_t j = blockIdx.x;
    const int lane = threadIdx.x;
    const int64_t c0 = cand_indptr[j];
    const int m = (int)(cand_indptr[j + 1] - c0);
    int s[4];
    double q[4], w[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int r = lane + 32 * t;
        s[t] = r < m ? cand_indices[c0 + r] : 0;
        if (r < m) ids[r] = s[t];
        q[t] = r < m ? (double)G[j * n + s[t]] : 0.0;   // b = G[S_j, j] = G[j, S_j]
        w[t] = 0.0;
    }
    __syncwarp();
#pragma unroll 4
    for (int p = 0; p < m; ++p) {
        const int* grow = G + (int64_t)ids[p] * n;
#pragma unroll
        for (int t = 0; t < 4; ++t)
            if (lane + 32 * t < m) Gs[p * m + lane + 32 * t] = grow[s[t]];
    }
    __syncwarp();

    int sweep = 0;
    bool done = false;
    while (!done) {
        ++sweep;
        double d = 0.0, wm = 0.0;
        unsigned act[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) act[t] = __ballot_sync(0xffffffffu, lane + 32 * t < m && (w[t] != 0.0 || q[t] > l1));
        for (int p = sl_next(act, 0); p < m; p = sl_next(act, p + 1)) {
            const int tp = p >> 5, src = p & 31;
            const double qp = __shfl_sync(0xffffffffu, sl_pick(q, tp), src);
            const double old = __shfl_sync(0xffffffffu, sl_pick(w, tp), src);
            const double gpp = (double)Gs[p * m + p];
            const double z = __dadd_rn(qp, __dmul_rn(gpp, old));
            const double nw = z > l1 ? __ddiv_rn(__dsub_rn(z, l1), __dadd_rn(gpp, l2)) : 0.0;
            const double delta = __dsub_rn(nw, old);
            if (nw != old) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const int r = lane + 32 * t;
                    if (r < m) q[t] = __dsub_rn(q[t], __dmul_rn((double)Gs[p * m + r], delta));
                    if (t == tp && lane == src) w[t] = nw;
                }
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    act[t] = __ballot_sync(0xffffffffu, lane + 32 * t < m && (w[t] != 0.0 || q[t] > l1));
            }
            const double ad = fabs(delta), an = fabs(nw);
            d = ad > d ? ad : d;
            wm = an > wm ? an : wm;
        }
        done = wm == 0.0 || d <= __dmul_rn(tol, wm) || sweep >= max_iter;
    }

    int base = 0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const bool pos = lane + 32 * t < m && w[t] > 0.0;
        const unsigned mk = __ballot_sync(0xffffffffu, pos);
        if (pos) {
            const int64_t at = j * kk + base + __popc(mk & ((1u << lane) - 1u));
            st_idx[at] = s[t];
            st_val[at] = w[t];
        }
        base += __popc(mk);
    }
    if (lane == 0) {
        cnt[j] = base;
        sweeps[j] = sweep;
    }
}

size_t slim_smem_bytes(int kk) { return ((size_t)kk * kk + SL_MAX) * sizeof(int); }

struct SlimLayout {
    size_t G, st_idx, st_val, cnt, total;
};

SlimLayout slim_layout(int64_t n, int kk) {
    SlimLayout L;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t at = off; off += align_up(bytes, 256); return at; };
    L.G = take((size_t)n * (size_t)n * 4);
    L.st_idx = take((size_t)n * kk * 4);
    L.st_val = take((size_t)n * kk * 8);
    L.cnt = take((size_t)n * 8);
    L.total = off;
    return L;
}

bool slim_finite_nonneg(double x) { return x >= 0.0 && x <= 1.7976931348623157e308; }

// ---- RP3beta (DESIGN.md 4.9): S_ab = sum over the common users u of a and b, ascending, of du[u], then
// W'_ab = (ra[a] S_ab) cb[b] and the top-k per row. The S tile is userknn_score_tile_kernel's score tile for "users"
// = items, "neighbours" = the users of the item (P^T, values du[u]) and "X" = P with every value 1.0f, so each
// product is du[u] exactly and each S_ab is summed from +0.0 in ascending u, one CTA per row, without atomics.

// nb_val[e] = du[pt_indices[e]] (the per-entry walk weights) and one[e] = 1.0f (the values of P)
__global__ __launch_bounds__(KN_THREADS) void rp3_gather_kernel(const int32_t* __restrict__ pt_indices, int64_t nnz,
                                                                const double* __restrict__ du,
                                                                double* __restrict__ nb_val, float* __restrict__ one) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        nb_val[e] = du[pt_indices[e]];
        one[e] = 1.0f;
    }
}

// chain[a] = sum over the users u of a of ceil(deg_u / KN_THREADS): the barrier steps of tile row a in
// userknn_score_tile_kernel. One warp per item.
__global__ __launch_bounds__(KN_THREADS) void rp3_chain_kernel(const int64_t* __restrict__ p_indptr,
                                                               const int64_t* __restrict__ pt_indptr,
                                                               const int32_t* __restrict__ pt_indices, int64_t n,
                                                               int64_t* __restrict__ chain) {
    const int64_t a = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (a >= n) return;
    const int lane = threadIdx.x & 31;
    int64_t s = 0;
    for (int64_t t = pt_indptr[a] + lane; t < pt_indptr[a + 1]; t += 32) {
        const int32_t u = pt_indices[t];
        s += (p_indptr[u + 1] - p_indptr[u] + KN_THREADS - 1) / KN_THREADS;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) chain[a] = s;
}

// order[rank(a)] = a with rank(a) = #{b : chain[b] > chain[a] or (chain[b] == chain[a] and b < a)}: the items by
// descending chain, ties by id (a permutation, so the same order every run). n^2 comparisons against KN_THREADS-item
// chunks staged in shared memory; training writes n^2 tile entries anyway.
__global__ __launch_bounds__(KN_THREADS) void rp3_order_kernel(const int64_t* __restrict__ chain, int64_t n,
                                                               int64_t* __restrict__ order) {
    __shared__ int64_t s_chain[KN_THREADS];
    const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t ca = a < n ? chain[a] : 0;
    int64_t rank = 0;
    for (int64_t b0 = 0; b0 < n; b0 += KN_THREADS) {
        __syncthreads();
        if (b0 + threadIdx.x < n) s_chain[threadIdx.x] = chain[b0 + threadIdx.x];
        __syncthreads();
        const int m = (int)(n - b0 < KN_THREADS ? n - b0 : KN_THREADS);
        for (int q = 0; q < m; ++q) {
            const int64_t cb = s_chain[q];
            rank += cb > ca || (cb == ca && b0 + q < a);
        }
    }
    if (a < n) order[rank] = a;
}

// S[r][b] = W'(a, b) for a = order[a0 + r]: (ra[a] S_ab) cb[b], rounded to nearest; self and S_ab = 0 (no common user)
// get RankKey<double>::excluded()
__global__ __launch_bounds__(KN_THREADS) void rp3_weight_kernel(double* __restrict__ S,
                                                                const int64_t* __restrict__ order, int64_t a0,
                                                                int64_t n, const double* __restrict__ ra,
                                                                const double* __restrict__ cb) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const int64_t r = blockIdx.y, a = order[a0 + r], e = r * n + b;
    const double s = S[e];
    S[e] = s > 0.0 && b != a ? __dmul_rn(__dmul_rn(ra[a], s), cb[b]) : RankKey<double>::excluded();
}

// One CTA per block row: selection row r into staging row order[a0 + r]
__global__ __launch_bounds__(KN_THREADS) void rp3_sort_rows_kernel(const int64_t* __restrict__ ids,
                                                                   const double* __restrict__ vals, int kk,
                                                                   const int64_t* __restrict__ order, int64_t a0,
                                                                   int32_t* __restrict__ st_idx,
                                                                   double* __restrict__ st_val,
                                                                   int64_t* __restrict__ cnt) {
    knn_sort_row(ids, vals, kk, blockIdx.x, order[a0 + blockIdx.x], st_idx, st_val, cnt);
}

struct Rp3Layout {
    size_t S, ids, vals, st_idx, st_val, cnt, chain, order, nb_val, one, total;
};

Rp3Layout rp3_layout(int64_t n, int64_t nnz, int kk) {
    const size_t B = (size_t)knn_batch(n, n);
    Rp3Layout L;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t at = off; off += align_up(bytes, 256); return at; };
    L.S = take(B * n * 8);
    L.ids = take(B * kk * 8);
    L.vals = take(B * kk * 8);
    L.st_idx = take((size_t)n * kk * 4);
    L.st_val = take((size_t)n * kk * 8);
    L.cnt = take((size_t)n * 8);
    L.chain = take((size_t)n * 8);
    L.order = take((size_t)n * 8);
    L.nb_val = take((size_t)nnz * 8);
    L.one = take((size_t)nnz * 4);
    L.total = off;
    return L;
}

int check_knn_args(const char* name, int64_t n, int k, int similarity, double shrink) {
    WMF_REQUIRE(n > 0 && n < (1ll << 31), "%s: n=%lld outside 1..2^31-1", name, (long long)n);
    WMF_REQUIRE(k >= 1 && k <= TK_MAX, "%s: k=%d outside 1..%d", name, k, TK_MAX);
    WMF_REQUIRE(similarity == WMF_KNN_COSINE || similarity == WMF_KNN_JACCARD || similarity == WMF_KNN_CONDITIONAL,
                "%s: unknown similarity %d", name, similarity);
    WMF_REQUIRE(shrink >= 0.0 && shrink <= 1.7976931348623157e308, "%s: shrink=%g is not finite and >= 0", name, shrink);
    return WMF_OK;
}

}  // namespace

}  // namespace wmf

using namespace wmf;

extern "C" {

size_t wmf_knn_train_workspace_bytes(int64_t n, int k) {
    if (n <= 0 || n >= (1ll << 31) || k < 1 || k > TK_MAX) return 0;
    return train_layout(n, n, (int)(k < n ? k : n), (size_t)knn_batch(n, n)).total;
}

int wmf_knn_train(const int64_t* x_indptr, const int32_t* x_indices, int64_t rows, const int64_t* xt_indptr,
                  const int32_t* xt_indices, int64_t n, int k, int similarity, double shrink, int64_t* w_indptr,
                  int32_t* w_indices, double* w_data, void* ws, size_t ws_bytes, void* stream) {
    if (int rc = check_knn_args("wmf_knn_train", n, k, similarity, shrink)) return rc;
    WMF_REQUIRE(rows >= 0, "wmf_knn_train: rows=%lld < 0", (long long)rows);
    WMF_REQUIRE(x_indptr && xt_indptr && w_indptr && w_indices && w_data, "wmf_knn_train: null argument");
    const size_t need = wmf_knn_train_workspace_bytes(n, k);
    if (ws == nullptr || ws_bytes < need) {
        set_error("wmf_knn_train: workspace %zu < %zu", ws_bytes, need);
        return WMF_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int kk = (int)(k < n ? k : n);
    const TrainLayout L = train_layout(n, n, kk, (size_t)knn_batch(n, n));
    char* base = reinterpret_cast<char*>(ws);
    int* C = reinterpret_cast<int*>(base + L.C);
    double* S = reinterpret_cast<double*>(base + L.S);
    int64_t* ids = reinterpret_cast<int64_t*>(base + L.ids);
    double* vals = reinterpret_cast<double*>(base + L.vals);
    int32_t* st_idx = reinterpret_cast<int32_t*>(base + L.st_idx);
    double* st_val = reinterpret_cast<double*>(base + L.st_val);
    int64_t* cnt = reinterpret_cast<int64_t*>(base + L.cnt);
    const int64_t bmax = knn_batch(n, n);
    const unsigned cooc_grid = (unsigned)sm_count() * 8;
    for (int64_t a0 = 0; a0 < n; a0 += bmax) {
        const int B = (int)(n - a0 < bmax ? n - a0 : bmax);
        WMF_CUDA(cudaMemsetAsync(C, 0, (size_t)B * n * 4, st));
        if (rows > 0) {
            knn_cooc_kernel<<<cooc_grid, KN_THREADS, 0, st>>>(x_indptr, x_indices, xt_indptr, xt_indices, n, a0, B, C);
            WMF_LAUNCH_CHECK("knn_cooc_kernel");
        }
        knn_similarity_kernel<<<dim3((unsigned)((n + KN_THREADS - 1) / KN_THREADS), (unsigned)B), KN_THREADS, 0, st>>>(
            C, xt_indptr, n, a0, similarity, shrink, S);
        WMF_LAUNCH_CHECK("knn_similarity_kernel");
        const int rc = select_topk_double(nullptr, 0, B, nullptr, nullptr, S, n, kk, ids, vals, st, true);
        if (rc) return rc;
        knn_sort_rows_kernel<<<(unsigned)B, KN_THREADS, 0, st>>>(ids, vals, kk, a0, st_idx, st_val, cnt);
        WMF_LAUNCH_CHECK("knn_sort_rows_kernel");
    }
    knn_scan_kernel<<<1, KN_THREADS, 0, st>>>(cnt, n, w_indptr);
    WMF_LAUNCH_CHECK("knn_scan_kernel");
    knn_compact_kernel<<<(unsigned)((n + KN_THREADS / 32 - 1) / (KN_THREADS / 32)), KN_THREADS, 0, st>>>(
        st_idx, st_val, kk, n, w_indptr, w_indices, w_data);
    WMF_LAUNCH_CHECK("knn_compact_kernel");
    return WMF_OK;
}

int wmf_knn_predict(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data, const int64_t* w_indptr,
                    const int32_t* w_indices, const double* w_data, const int64_t* users, int64_t user_stride,
                    const int64_t* items, int64_t count, double* out, void* stream) {
    WMF_REQUIRE(count >= 0 && user_stride >= 0, "wmf_knn_predict: bad arguments");
    if (count == 0) return WMF_OK;
    WMF_REQUIRE(x_indptr && w_indptr && users && items && out, "wmf_knn_predict: null argument");
    knn_predict_kernel<<<(unsigned)((count + KN_THREADS - 1) / KN_THREADS), KN_THREADS, 0, (cudaStream_t)stream>>>(
        x_indptr, x_indices, x_data, w_indptr, w_indices, w_data, users, user_stride, items, count, out);
    WMF_LAUNCH_CHECK("knn_predict_kernel");
    return WMF_OK;
}

size_t wmf_knn_score_topk_workspace_bytes(int64_t nu, int64_t n, int topn) {
    (void)topn;
    return score_topk_double_workspace_bytes(nu, n, knn_batch);
}

int wmf_knn_score_topk(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data, const int64_t* w_indptr,
                       const int32_t* w_indices, const double* w_data, int64_t n, const int64_t* users, int64_t nu,
                       const int64_t* ex_indptr, const int32_t* ex_indices, int topn, int64_t* out_ids,
                       double* out_scores, void* ws, size_t ws_bytes, void* stream) {
    return score_topk_double("wmf_knn_score_topk", x_indptr && w_indptr, knn_batch, n, users, nu, ex_indptr, ex_indices,
                             topn, out_ids, out_scores, ws, ws_bytes, stream,
                             [&](int64_t u0, int ub, double* S, cudaStream_t st) {
        WMF_CUDA(cudaMemsetAsync(S, 0, (size_t)ub * n * sizeof(double), st));
        knn_score_tile_kernel<<<(unsigned)((ub + KN_THREADS / 32 - 1) / (KN_THREADS / 32)), KN_THREADS, 0, st>>>(
            x_indptr, x_indices, x_data, w_indptr, w_indices, w_data, n, users, u0, ub, S);
        WMF_LAUNCH_CHECK("knn_score_tile_kernel");
        return WMF_OK;
    });
}

int wmf_userknn_predict(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data,
                        const int64_t* nb_indptr, const int32_t* nb_indices, const double* nb_data,
                        const int64_t* users, int64_t user_stride, const int64_t* items, int64_t count, double* out,
                        void* stream) {
    WMF_REQUIRE(count >= 0 && user_stride >= 0, "wmf_userknn_predict: bad arguments");
    if (count == 0) return WMF_OK;
    WMF_REQUIRE(x_indptr && nb_indptr && users && items && out, "wmf_userknn_predict: null argument");
    userknn_predict_kernel<<<(unsigned)((count + KN_THREADS - 1) / KN_THREADS), KN_THREADS, 0, (cudaStream_t)stream>>>(
        x_indptr, x_indices, x_data, nb_indptr, nb_indices, nb_data, users, user_stride, items, count, out);
    WMF_LAUNCH_CHECK("userknn_predict_kernel");
    return WMF_OK;
}

size_t wmf_userknn_score_topk_workspace_bytes(int64_t nu, int64_t n, int topn) {
    (void)topn;
    return score_topk_double_workspace_bytes(nu, n, knn_batch);
}

int wmf_userknn_score_topk(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data,
                           const int64_t* nb_indptr, const int32_t* nb_indices, const double* nb_data, int64_t n,
                           const int64_t* users, int64_t nu, const int64_t* ex_indptr, const int32_t* ex_indices,
                           int topn, int64_t* out_ids, double* out_scores, void* ws, size_t ws_bytes, void* stream) {
    return score_topk_double("wmf_userknn_score_topk", x_indptr && nb_indptr, knn_batch, n, users, nu, ex_indptr,
                             ex_indices, topn, out_ids, out_scores, ws, ws_bytes, stream,
                             [&](int64_t u0, int ub, double* S, cudaStream_t st) {
        WMF_CUDA(cudaMemsetAsync(S, 0, (size_t)ub * n * sizeof(double), st));
        userknn_score_tile_kernel<<<(unsigned)ub, KN_THREADS, 0, st>>>(x_indptr, x_indices, x_data, nb_indptr,
                                                                      nb_indices, nb_data, n, users, u0, S);
        WMF_LAUNCH_CHECK("userknn_score_tile_kernel");
        return WMF_OK;
    });
}

size_t wmf_userknn_fold_in_workspace_bytes(int64_t nq, int64_t m, int k) {
    if (nq <= 0 || nq >= (1ll << 31) || m <= 0 || m >= (1ll << 31) || k < 1 || k > TK_MAX) return 0;
    return train_layout(nq, m, (int)(k < m ? k : m), (size_t)fold_in_batch(nq, m)).total;
}

int wmf_userknn_fold_in(const int64_t* q_indptr, const int32_t* q_indices, int64_t nq, const int64_t* xt_indptr,
                        const int32_t* xt_indices, int64_t n_items, const int64_t* x_indptr, int64_t m, int k,
                        int similarity, double shrink, int64_t* out_indptr, int32_t* out_indices, double* out_data,
                        void* ws, size_t ws_bytes, void* stream) {
    if (int rc = check_knn_args("wmf_userknn_fold_in", m, k, similarity, shrink)) return rc;
    WMF_REQUIRE(nq > 0 && nq < (1ll << 31), "wmf_userknn_fold_in: nq=%lld outside 1..2^31-1", (long long)nq);
    WMF_REQUIRE(n_items >= 0, "wmf_userknn_fold_in: n_items=%lld < 0", (long long)n_items);
    WMF_REQUIRE(q_indptr && xt_indptr && x_indptr && out_indptr && out_indices && out_data,
                "wmf_userknn_fold_in: null argument");
    const size_t need = wmf_userknn_fold_in_workspace_bytes(nq, m, k);
    if (ws == nullptr || ws_bytes < need) {
        set_error("wmf_userknn_fold_in: workspace %zu < %zu", ws_bytes, need);
        return WMF_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int kk = (int)(k < m ? k : m);
    const int64_t bmax = fold_in_batch(nq, m);
    const TrainLayout L = train_layout(nq, m, kk, (size_t)bmax);
    char* base = reinterpret_cast<char*>(ws);
    int* C = reinterpret_cast<int*>(base + L.C);
    double* S = reinterpret_cast<double*>(base + L.S);
    int64_t* ids = reinterpret_cast<int64_t*>(base + L.ids);
    double* vals = reinterpret_cast<double*>(base + L.vals);
    int32_t* st_idx = reinterpret_cast<int32_t*>(base + L.st_idx);
    double* st_val = reinterpret_cast<double*>(base + L.st_val);
    int64_t* cnt = reinterpret_cast<int64_t*>(base + L.cnt);
    const unsigned cooc_grid = (unsigned)sm_count() * 8;
    for (int64_t r0 = 0; r0 < nq; r0 += bmax) {
        const int B = (int)(nq - r0 < bmax ? nq - r0 : bmax);
        WMF_CUDA(cudaMemsetAsync(C, 0, (size_t)B * m * 4, st));
        if (n_items > 0) {   // the new rows are the "X^T" of the counts (rows -> items), the training X^T their "X"
            knn_cooc_kernel<<<cooc_grid, KN_THREADS, 0, st>>>(xt_indptr, xt_indices, q_indptr, q_indices, m, r0, B, C);
            WMF_LAUNCH_CHECK("knn_cooc_kernel");
        }
        userknn_cross_similarity_kernel<<<dim3((unsigned)((m + KN_THREADS - 1) / KN_THREADS), (unsigned)B), KN_THREADS,
                                          0, st>>>(C, q_indptr, x_indptr, m, r0, similarity, shrink, S);
        WMF_LAUNCH_CHECK("userknn_cross_similarity_kernel");
        const int rc = select_topk_double(nullptr, 0, B, nullptr, nullptr, S, m, kk, ids, vals, st, true);
        if (rc) return rc;
        knn_sort_rows_kernel<<<(unsigned)B, KN_THREADS, 0, st>>>(ids, vals, kk, r0, st_idx, st_val, cnt);
        WMF_LAUNCH_CHECK("knn_sort_rows_kernel");
    }
    knn_scan_kernel<<<1, KN_THREADS, 0, st>>>(cnt, nq, out_indptr);
    WMF_LAUNCH_CHECK("knn_scan_kernel");
    knn_compact_kernel<<<(unsigned)((nq + KN_THREADS / 32 - 1) / (KN_THREADS / 32)), KN_THREADS, 0, st>>>(
        st_idx, st_val, kk, nq, out_indptr, out_indices, out_data);
    WMF_LAUNCH_CHECK("knn_compact_kernel");
    return WMF_OK;
}

size_t wmf_slim_train_workspace_bytes(int64_t n, int k) {
    if (n <= 0 || n > (1ll << 30) || k < 1 || k > SL_MAX) return 0;
    return slim_layout(n, (int)(k < n ? k : n)).total;
}

int wmf_slim_train(const int64_t* x_indptr, const int32_t* x_indices, int64_t rows, const int64_t* xt_indptr,
                   const int32_t* xt_indices, int64_t n, const int64_t* cand_indptr, const int32_t* cand_indices, int k,
                   double l1, double l2, int max_iter, double tol, int64_t* wt_indptr, int32_t* wt_indices,
                   double* wt_data, int32_t* sweeps, void* ws, size_t ws_bytes, void* stream) {
    WMF_REQUIRE(n > 0 && n <= (1ll << 30), "wmf_slim_train: n=%lld outside 1..2^30", (long long)n);
    WMF_REQUIRE(k >= 1 && k <= SL_MAX, "wmf_slim_train: k=%d outside 1..%d", k, SL_MAX);
    WMF_REQUIRE(slim_finite_nonneg(l1), "wmf_slim_train: l1=%g is not finite and >= 0", l1);
    WMF_REQUIRE(slim_finite_nonneg(l2), "wmf_slim_train: l2=%g is not finite and >= 0", l2);
    WMF_REQUIRE(max_iter >= 1, "wmf_slim_train: max_iter=%d < 1", max_iter);
    WMF_REQUIRE(slim_finite_nonneg(tol), "wmf_slim_train: tol=%g is not finite and >= 0", tol);
    WMF_REQUIRE(rows >= 0, "wmf_slim_train: rows=%lld < 0", (long long)rows);
    WMF_REQUIRE(x_indptr && xt_indptr && cand_indptr && wt_indptr && wt_indices && wt_data && sweeps,
                "wmf_slim_train: null argument");
    const size_t need = wmf_slim_train_workspace_bytes(n, k);
    if (ws == nullptr || ws_bytes < need) {
        set_error("wmf_slim_train: workspace %zu < %zu", ws_bytes, need);
        return WMF_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int kk = (int)(k < n ? k : n);
    const SlimLayout L = slim_layout(n, kk);
    char* base = reinterpret_cast<char*>(ws);
    int* G = reinterpret_cast<int*>(base + L.G);
    int32_t* st_idx = reinterpret_cast<int32_t*>(base + L.st_idx);
    double* st_val = reinterpret_cast<double*>(base + L.st_val);
    int64_t* cnt = reinterpret_cast<int64_t*>(base + L.cnt);
    WMF_CUDA(cudaMemsetAsync(G, 0, (size_t)n * (size_t)n * 4, st));
    if (rows > 0) {
        knn_cooc_kernel<<<(unsigned)sm_count() * 8, KN_THREADS, 0, st>>>(x_indptr, x_indices, xt_indptr, xt_indices, n,
                                                                         0, (int)n, G);
        WMF_LAUNCH_CHECK("knn_cooc_kernel");
    }
    const size_t smem = slim_smem_bytes(kk);
    WMF_CUDA(cudaFuncSetAttribute(slim_cd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    slim_cd_kernel<<<(unsigned)n, 32, smem, st>>>(G, n, cand_indptr, cand_indices, kk, l1, l2, max_iter, tol, st_idx,
                                                  st_val, cnt, sweeps);
    WMF_LAUNCH_CHECK("slim_cd_kernel");
    knn_scan_kernel<<<1, KN_THREADS, 0, st>>>(cnt, n, wt_indptr);
    WMF_LAUNCH_CHECK("knn_scan_kernel");
    knn_compact_kernel<<<(unsigned)((n + KN_THREADS / 32 - 1) / (KN_THREADS / 32)), KN_THREADS, 0, st>>>(
        st_idx, st_val, kk, n, wt_indptr, wt_indices, wt_data);
    WMF_LAUNCH_CHECK("knn_compact_kernel");
    return WMF_OK;
}

size_t wmf_rp3beta_train_workspace_bytes(int64_t n, int64_t nnz, int k) {
    if (n <= 0 || n >= (1ll << 31) || nnz < 0 || nnz >= (1ll << 40) || k < 1 || k > TK_MAX) return 0;
    return rp3_layout(n, nnz, (int)(k < n ? k : n)).total;
}

int wmf_rp3beta_train(const int64_t* p_indptr, const int32_t* p_indices, int64_t rows, const int64_t* pt_indptr,
                      const int32_t* pt_indices, int64_t n, int64_t nnz, const double* du, const double* ra,
                      const double* cb, int k, int64_t* w_indptr, int32_t* w_indices, double* w_data, void* ws,
                      size_t ws_bytes, void* stream) {
    WMF_REQUIRE(n > 0 && n < (1ll << 31), "wmf_rp3beta_train: n=%lld outside 1..2^31-1", (long long)n);
    WMF_REQUIRE(k >= 1 && k <= TK_MAX, "wmf_rp3beta_train: k=%d outside 1..%d", k, TK_MAX);
    WMF_REQUIRE(rows >= 0, "wmf_rp3beta_train: rows=%lld < 0", (long long)rows);
    WMF_REQUIRE(nnz >= 0 && nnz < (1ll << 40), "wmf_rp3beta_train: nnz=%lld outside 0..2^40-1", (long long)nnz);
    WMF_REQUIRE(p_indptr && pt_indptr && (du || rows == 0) && ra && cb && w_indptr && w_indices && w_data &&
                    ((p_indices && pt_indices) || nnz == 0),
                "wmf_rp3beta_train: null argument");
    const size_t need = wmf_rp3beta_train_workspace_bytes(n, nnz, k);
    if (ws == nullptr || ws_bytes < need) {
        set_error("wmf_rp3beta_train: workspace %zu < %zu", ws_bytes, need);
        return WMF_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int kk = (int)(k < n ? k : n);
    const Rp3Layout L = rp3_layout(n, nnz, kk);
    char* base = reinterpret_cast<char*>(ws);
    double* S = reinterpret_cast<double*>(base + L.S);
    int64_t* ids = reinterpret_cast<int64_t*>(base + L.ids);
    double* vals = reinterpret_cast<double*>(base + L.vals);
    int32_t* st_idx = reinterpret_cast<int32_t*>(base + L.st_idx);
    double* st_val = reinterpret_cast<double*>(base + L.st_val);
    int64_t* cnt = reinterpret_cast<int64_t*>(base + L.cnt);
    int64_t* chain = reinterpret_cast<int64_t*>(base + L.chain);
    int64_t* order = reinterpret_cast<int64_t*>(base + L.order);
    double* nb_val = reinterpret_cast<double*>(base + L.nb_val);
    float* one = reinterpret_cast<float*>(base + L.one);
    if (nnz > 0) {
        rp3_gather_kernel<<<(unsigned)sm_count() * 8, KN_THREADS, 0, st>>>(pt_indices, nnz, du, nb_val, one);
        WMF_LAUNCH_CHECK("rp3_gather_kernel");
    }
    rp3_chain_kernel<<<(unsigned)((n + KN_THREADS / 32 - 1) / (KN_THREADS / 32)), KN_THREADS, 0, st>>>(
        p_indptr, pt_indptr, pt_indices, n, chain);
    WMF_LAUNCH_CHECK("rp3_chain_kernel");
    rp3_order_kernel<<<(unsigned)((n + KN_THREADS - 1) / KN_THREADS), KN_THREADS, 0, st>>>(chain, n, order);
    WMF_LAUNCH_CHECK("rp3_order_kernel");
    const int64_t bmax = knn_batch(n, n);
    for (int64_t a0 = 0; a0 < n; a0 += bmax) {
        const int B = (int)(n - a0 < bmax ? n - a0 : bmax);
        WMF_CUDA(cudaMemsetAsync(S, 0, (size_t)B * n * sizeof(double), st));
        userknn_score_tile_kernel<<<(unsigned)B, KN_THREADS, 0, st>>>(p_indptr, p_indices, one, pt_indptr, pt_indices,
                                                                     nb_val, n, order, a0, S);
        WMF_LAUNCH_CHECK("userknn_score_tile_kernel");
        rp3_weight_kernel<<<dim3((unsigned)((n + KN_THREADS - 1) / KN_THREADS), (unsigned)B), KN_THREADS, 0, st>>>(
            S, order, a0, n, ra, cb);
        WMF_LAUNCH_CHECK("rp3_weight_kernel");
        const int rc = select_topk_double(nullptr, 0, B, nullptr, nullptr, S, n, kk, ids, vals, st, true);
        if (rc) return rc;
        rp3_sort_rows_kernel<<<(unsigned)B, KN_THREADS, 0, st>>>(ids, vals, kk, order, a0, st_idx, st_val, cnt);
        WMF_LAUNCH_CHECK("rp3_sort_rows_kernel");
    }
    knn_scan_kernel<<<1, KN_THREADS, 0, st>>>(cnt, n, w_indptr);
    WMF_LAUNCH_CHECK("knn_scan_kernel");
    knn_compact_kernel<<<(unsigned)((n + KN_THREADS / 32 - 1) / (KN_THREADS / 32)), KN_THREADS, 0, st>>>(
        st_idx, st_val, kk, n, w_indptr, w_indices, w_data);
    WMF_LAUNCH_CHECK("knn_compact_kernel");
    return WMF_OK;
}

}  // extern "C"
