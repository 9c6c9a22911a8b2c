// Shared by the exact (score.cu) and tensor-core (score_tc.cu) ranking paths, and by the EASE (ease.cu) and ItemKNN
// (knn.cu) models.
#pragma once
#include "common.cuh"

namespace wmf {

constexpr int TK_MAX = 1024;  // largest topn the selection kernel sorts in shared memory

// order-preserving map float -> uint32 (larger float -> larger key)
__device__ __forceinline__ uint32_t order_key(float x) {
    uint32_t b = __float_as_uint(x);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// order-preserving map double -> uint64
__device__ __forceinline__ unsigned long long order_key(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}

// What the selection kernel (topk_rows_kernel) sorts for each score type. The all-ones score (`excluded()`) maps to
// key 0, below every other score. An Entry packs the order key with 0xFFFFFFFF - position, so that the larger entry
// is the larger score and, among equal scores, the lower position.
template <typename T> struct RankKey;

template <> struct RankKey<float> {
    using Key = uint32_t;
    using Entry = unsigned long long;
    static constexpr int BITS = 32;
    __device__ static float excluded() { return __uint_as_float(0xFFFFFFFFu); }
    __device__ static Entry entry(Key k, uint32_t pos) {
        return ((unsigned long long)k << 32) | (unsigned long long)(0xFFFFFFFFu - pos);
    }
    __device__ static bool less(Entry a, Entry b) { return a < b; }
    __device__ static uint32_t pos(Entry e) { return 0xFFFFFFFFu - (uint32_t)(e & 0xFFFFFFFFull); }
    __device__ static Key key(Entry e) { return (Key)(e >> 32); }
};

template <> struct RankKey<double> {
    using Key = unsigned long long;
    struct Entry {
        unsigned long long k;
        uint32_t p;  // 0xFFFFFFFF - position
    };
    static constexpr int BITS = 64;
    __device__ static double excluded() { return __longlong_as_double(-1ll); }
    __device__ static Entry entry(Key k, uint32_t pos) { return Entry{k, 0xFFFFFFFFu - pos}; }
    __device__ static bool less(Entry a, Entry b) { return a.k < b.k || (a.k == b.k && a.p < b.p); }
    __device__ static uint32_t pos(Entry e) { return 0xFFFFFFFFu - e.p; }
    __device__ static Key key(Entry e) { return e.k; }
};

// Exact selection over a [ub x ni] tile of double scores S (row r: user users[u_begin + r]), the kernels of the exact
// ranking path instantiated for double (score.cu). ex_indptr (nullable) / ex_indices: the exclusion CSR by user id.
// out_ids / out_scores (nullable) [ub x topn]; topn in 1..min(ni, TK_MAX). `marked`: S already holds
// RankKey<double>::excluded() entries of its own (users may then be null when ex_indptr is), which, like excluded
// items, are reported as id -1 when a row has fewer than topn other entries.
int select_topk_double(const int64_t* users, int64_t u_begin, int ub, const int64_t* ex_indptr, const int32_t* ex_indices,
                       double* S, int64_t ni, int topn, int64_t* out_ids, double* out_scores, cudaStream_t st,
                       bool marked = false);

// Bytes of the [user_batch(nu, n) x n] double score tile that score_topk_double needs; 0 when nu or n is out of range.
inline size_t score_topk_double_workspace_bytes(int64_t nu, int64_t n, int64_t (*user_batch)(int64_t, int64_t)) {
    if (nu <= 0 || n <= 0 || n >= (1ll << 31)) return 0;
    return align_up((size_t)user_batch(nu, n) * (size_t)n * sizeof(double), 1024);
}

// The exact double top-N over all n items of a model that scores users tile by tile (wmf_ease_score_topk,
// wmf_knn_score_topk; `name` prefixes the messages). The checks run in a fixed order: n, nu, topn (WMF_ERR_UNSUPPORTED),
// nu == 0 returns WMF_OK before any pointer is looked at, then the pointers (`inputs_ok`: the model's own inputs are
// non-null) and the workspace. Then, for each batch of ub <= user_batch(nu, n) users from u0, score_tile(u0, ub, S, st)
// writes their [ub x n] scores into the workspace S and returns a WMF_* code, and select_topk_double ranks them.
template <typename ScoreTile>
int score_topk_double(const char* name, bool inputs_ok, int64_t (*user_batch)(int64_t, int64_t), int64_t n,
                      const int64_t* users, int64_t nu, const int64_t* ex_indptr, const int32_t* ex_indices, int topn,
                      int64_t* out_ids, double* out_scores, void* ws, size_t ws_bytes, void* stream,
                      ScoreTile score_tile) {
    WMF_REQUIRE(n > 0 && n < (1ll << 31), "%s: n=%lld outside 1..2^31-1", name, (long long)n);
    WMF_REQUIRE(nu >= 0, "%s: nu=%lld < 0", name, (long long)nu);
    if (topn < 1 || topn > n || topn > TK_MAX) {
        set_error("%s: topn=%d outside 1..min(n=%lld, %d)", name, topn, (long long)n, TK_MAX);
        return WMF_ERR_UNSUPPORTED;
    }
    if (nu == 0) return WMF_OK;
    WMF_REQUIRE(inputs_ok && users && out_ids, "%s: null argument", name);
    const size_t need = score_topk_double_workspace_bytes(nu, n, user_batch);
    if (ws == nullptr || ws_bytes < need) {
        set_error("%s: workspace %zu < %zu", name, ws_bytes, need);
        return WMF_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t ubatch = user_batch(nu, n);
    double* S = (double*)ws;
    for (int64_t u0 = 0; u0 < nu; u0 += ubatch) {
        const int ub = (int)((nu - u0) < ubatch ? (nu - u0) : ubatch);
        if (int rc = score_tile(u0, ub, S, st)) return rc;
        if (int rc = select_topk_double(users, u0, ub, ex_indptr, ex_indices, S, n, topn, out_ids + (size_t)u0 * topn,
                                        out_scores ? out_scores + (size_t)u0 * topn : nullptr, st))
            return rc;
    }
    return WMF_OK;
}

bool score_tc_supported(int64_t ni, int f, int bias, int topn);
size_t score_tc_workspace_bytes(int64_t nu, int64_t ni);
int64_t score_tc_user_batch(int64_t nu);
void score_tc_fixup_region(int64_t nu, int64_t ni, size_t* offset, size_t* bytes);
int score_topk_tc_batch(const int64_t* users, int64_t u0, int ub, int64_t ubatch, const int64_t* cand, int64_t ni,
                        const float* U, int64_t ldu, const float* V, int64_t ldv, int f, int bias, int topn,
                        int64_t* out_ids, float* out_scores, void* ws, bool first_batch, int** overflow_flag,
                        cudaStream_t st, const int64_t* ex_indptr, const int32_t* ex_indices, int* fixup_users);

}  // namespace wmf
