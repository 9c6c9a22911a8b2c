// N5: full-ranking quality of the top-N lists WMF.recommend returns (WMF.eval_ranking). No reference call site:
// the reference's only ranking measure is the sampled Recall@N of eval_topn (N2, eval_topn.cu).
//
// For user u with list r_1..r_K (item ids, -1 = padding, never a hit), T_u = the distinct column ids of row u of the
// test matrix with at least one stored non-zero value, and h_i = |{j <= i : r_j in T_u}|, each cutoff k gives
//   Precision@k = h_k / k                  Recall@k = h_k / |T_u|              HitRate@k = [h_k > 0]
//   NDCG@k = sum_{i<=k, r_i in T_u} 1/log2(i+1) / sum_{i=1}^{min(k,|T_u|)} 1/log2(i+1)
//   MAP@k  = sum_{i<=k, r_i in T_u} h_i / i / min(k, |T_u|)
// A user with T_u empty gets a NaN row and is left out of the means.
//
// topn_metrics_kernel: one warp per user. |T_u| is one lane-strided pass over the (sorted) test row: an entry counts
// when it is non-zero and no earlier entry of its run of equal ids is. The lanes then take the ranked positions 32 at a
// time; a position is a hit when a lower-bound binary search finds its id in the row and the run of equal ids holds a
// non-zero value. h_i is a ballot/popc prefix plus the hits of the earlier chunks. The DCG, AP and IDCG terms are
// doubles; a cutoff inside a chunk adds the masked butterfly sum of that chunk to the running totals of the chunks
// before it. Every sum runs in an order fixed by the data alone, so a user's row is bitwise reproducible and does not
// depend on which other users share the launch.
//
// The reduce adds the rows in blocks of REDUCE_ROWS users (a thread per value, rows in order), then one block adds the
// block partials in block order. The grid depends on nu alone: the sums are reproducible from run to run and do not
// depend on how the caller filled the per-user buffer.
#include "common.cuh"

namespace wmf {

constexpr int METRICS_THREADS = 256;
constexpr int METRICS_MAX_CUTS = 16;
constexpr int METRICS_PER_CUT = 5;  // Recall, Precision, NDCG, MAP, HitRate
constexpr int REDUCE_ROWS = 256;

struct TopnCuts {
    int k[METRICS_MAX_CUTS];     // ascending
    int slot[METRICS_MAX_CUTS];  // position of k[c] in the caller's list
    int n;
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// id in T_u: lower bound in the sorted row, then the run of equal ids for a non-zero value
__device__ __forceinline__ bool in_test_row(const int32_t* __restrict__ idx, const float* __restrict__ val,
                                            int64_t lo, int64_t hi, int64_t id) {
    int64_t a = lo, b = hi;
    while (a < b) {
        const int64_t m = (a + b) >> 1;
        if ((int64_t)idx[m] < id) a = m + 1; else b = m;
    }
    for (; a < hi && (int64_t)idx[a] == id; ++a)
        if (val[a] != 0.0f) return true;
    return false;
}

__global__ __launch_bounds__(METRICS_THREADS) void topn_metrics_kernel(
        const int64_t* __restrict__ ids, int64_t nu, int K, const int64_t* __restrict__ users,
        const int64_t* __restrict__ t_indptr, const int32_t* __restrict__ t_indices, const float* __restrict__ t_data,
        const TopnCuts cuts, double* __restrict__ per_user) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= nu) return;
    const int nk = cuts.n;
    double* out = per_user + w * (int64_t)(nk * METRICS_PER_CUT);
    const int64_t u = users[w];
    const int64_t lo = t_indptr[u], hi = t_indptr[u + 1];

    int t = 0;  // |T_u|
    for (int64_t e = lo + lane; e < hi; e += 32) {
        if (t_data[e] == 0.0f) continue;
        const int32_t id = t_indices[e];
        bool first = true;
        for (int64_t p = e - 1; p >= lo && t_indices[p] == id; --p)
            if (t_data[p] != 0.0f) { first = false; break; }
        t += first ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (t == 0) {
        for (int j = lane; j < nk * METRICS_PER_CUT; j += 32) out[j] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }

    const int64_t* r = ids + w * (int64_t)K;
    const int kmax = cuts.k[nk - 1];
    const unsigned le_mask = 0xffffffffu >> (31 - lane);  // lanes 0..lane
    int carry = 0;                                        // hits before the chunk
    double dcg = 0.0, ap = 0.0, idcg = 0.0;               // sums over the chunks before this one
    int c = 0;
    for (int base = 0; c < nk; base += 32) {
        const int i = base + lane + 1;  // 1-based position of this lane
        bool hit = false;
        if (i <= kmax) {
            const int64_t id = r[i - 1];
            hit = id >= 0 && in_test_row(t_indices, t_data, lo, hi, id);
        }
        const unsigned ball = __ballot_sync(0xffffffffu, hit);
        const double disc = i <= kmax ? 1.0 / log2((double)(i + 1)) : 0.0;
        const double g = hit ? disc : 0.0;
        const double a = hit ? (double)(carry + __popc(ball & le_mask)) / (double)i : 0.0;
        const double ig = i <= t ? disc : 0.0;
        for (; c < nk && cuts.k[c] <= base + 32; ++c) {  // cutoffs that end inside this chunk
            const int k = cuts.k[c];
            const bool in = i <= k;
            const double sg = dcg + warp_sum_d(in ? g : 0.0);
            const double sa = ap + warp_sum_d(in ? a : 0.0);
            const double si = idcg + warp_sum_d(in ? ig : 0.0);
            const int h = carry + __popc(ball & (0xffffffffu >> (32 - (k - base))));
            if (lane == 0) {
                double* o = out + cuts.slot[c] * METRICS_PER_CUT;
                o[0] = (double)h / (double)t;
                o[1] = (double)h / (double)k;
                o[2] = sg / si;
                o[3] = sa / (double)min(k, t);
                o[4] = h > 0 ? 1.0 : 0.0;
            }
        }
        carry += __popc(ball);
        dcg += warp_sum_d(g);
        ap += warp_sum_d(a);
        idcg += warp_sum_d(ig);
    }
}

// partial[b][c] = sum over the rows of block b (in order) whose value 0 is not NaN of value c; c == ncols counts them
__global__ void topn_metrics_partial_kernel(const double* __restrict__ per_user, int64_t nu, int ncols,
                                            double* __restrict__ partial) {
    const int c = threadIdx.x;
    if (c > ncols) return;
    const int64_t r0 = (int64_t)blockIdx.x * REDUCE_ROWS;
    const int64_t r1 = min(nu, r0 + REDUCE_ROWS);
    double s = 0.0;
    for (int64_t r = r0; r < r1; ++r) {
        const double* row = per_user + r * ncols;
        const double v0 = row[0];
        if (isnan(v0)) continue;
        s += c < ncols ? row[c] : 1.0;
    }
    partial[(int64_t)blockIdx.x * (ncols + 1) + c] = s;
}

__global__ void topn_metrics_final_kernel(const double* __restrict__ partial, int64_t nblocks, int ncols,
                                          double* __restrict__ sums) {
    const int c = threadIdx.x;
    if (c > ncols) return;
    double s = 0.0;
    for (int64_t b = 0; b < nblocks; ++b) s += partial[b * (ncols + 1) + c];
    sums[c] = s;
}

}  // namespace wmf

using namespace wmf;

extern "C" {

size_t wmf_topn_metrics_workspace_bytes(int64_t nu, int nk) {
    if (nu <= 0 || nk <= 0 || nk > METRICS_MAX_CUTS) return 0;
    const int64_t blocks = (nu + REDUCE_ROWS - 1) / REDUCE_ROWS;
    return (size_t)blocks * (size_t)(nk * METRICS_PER_CUT + 1) * sizeof(double);
}

int wmf_topn_metrics(const int64_t* ids, int64_t nu, int K, const int64_t* users, const int64_t* t_indptr,
                     const int32_t* t_indices, const float* t_data, const int32_t* ks_host, int nk, double* per_user,
                     void* stream) {
    WMF_REQUIRE(nu >= 0 && K > 0, "wmf_topn_metrics: bad sizes (nu=%lld, K=%d)", (long long)nu, K);
    WMF_REQUIRE(nk >= 1 && nk <= METRICS_MAX_CUTS, "wmf_topn_metrics: nk=%d outside [1, %d]", nk, METRICS_MAX_CUTS);
    WMF_REQUIRE(ks_host != nullptr, "wmf_topn_metrics: null cutoff list");
    TopnCuts cuts;
    cuts.n = nk;
    for (int j = 0; j < nk; ++j) {
        WMF_REQUIRE(ks_host[j] >= 1 && ks_host[j] <= K, "wmf_topn_metrics: cutoff %d outside [1, %d]", ks_host[j], K);
        for (int q = 0; q < j; ++q) WMF_REQUIRE(ks_host[q] != ks_host[j], "wmf_topn_metrics: cutoff %d given twice", ks_host[j]);
        int p = j;  // insertion into the ascending list
        while (p > 0 && cuts.k[p - 1] > ks_host[j]) { cuts.k[p] = cuts.k[p - 1]; cuts.slot[p] = cuts.slot[p - 1]; --p; }
        cuts.k[p] = ks_host[j];
        cuts.slot[p] = j;
    }
    if (nu == 0) return WMF_OK;
    WMF_REQUIRE(ids && users && t_indptr && t_indices && t_data && per_user, "wmf_topn_metrics: null pointer");
    const int64_t blocks = (nu * 32 + METRICS_THREADS - 1) / METRICS_THREADS;
    WMF_REQUIRE(blocks < (1ll << 31), "wmf_topn_metrics: too many users in one call (%lld)", (long long)nu);
    topn_metrics_kernel<<<(unsigned)blocks, METRICS_THREADS, 0, (cudaStream_t)stream>>>(
        ids, nu, K, users, t_indptr, t_indices, t_data, cuts, per_user);
    WMF_LAUNCH_CHECK("topn_metrics_kernel");
    return WMF_OK;
}

int wmf_topn_metrics_reduce(const double* per_user, int64_t nu, int nk, double* sums, void* ws, size_t ws_bytes,
                            void* stream) {
    WMF_REQUIRE(nu >= 0, "wmf_topn_metrics_reduce: bad sizes (nu=%lld)", (long long)nu);
    WMF_REQUIRE(nk >= 1 && nk <= METRICS_MAX_CUTS, "wmf_topn_metrics_reduce: nk=%d outside [1, %d]", nk,
                METRICS_MAX_CUTS);
    WMF_REQUIRE(sums != nullptr && (nu == 0 || per_user != nullptr), "wmf_topn_metrics_reduce: null pointer");
    const int ncols = nk * METRICS_PER_CUT;
    const int64_t blocks = (nu + REDUCE_ROWS - 1) / REDUCE_ROWS;
    const size_t need = wmf_topn_metrics_workspace_bytes(nu, nk);
    if (nu > 0 && (ws == nullptr || ws_bytes < need)) {
        set_error("wmf_topn_metrics_reduce: workspace %zu < %zu", ws_bytes, need);
        return WMF_ERR_WORKSPACE;
    }
    WMF_REQUIRE(blocks < (1ll << 31), "wmf_topn_metrics_reduce: too many users (%lld)", (long long)nu);
    cudaStream_t st = (cudaStream_t)stream;
    if (nu == 0) {
        WMF_CUDA(cudaMemsetAsync(sums, 0, (size_t)(ncols + 1) * sizeof(double), st));
        return WMF_OK;
    }
    const int threads = (ncols + 1 + 31) / 32 * 32;
    topn_metrics_partial_kernel<<<(unsigned)blocks, threads, 0, st>>>(per_user, nu, ncols, (double*)ws);
    WMF_LAUNCH_CHECK("topn_metrics_partial_kernel");
    topn_metrics_final_kernel<<<1, threads, 0, st>>>((const double*)ws, blocks, ncols, sums);
    WMF_LAUNCH_CHECK("topn_metrics_final_kernel");
    return WMF_OK;
}

}  // extern "C"
