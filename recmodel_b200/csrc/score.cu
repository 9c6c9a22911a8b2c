// K4 + K5: top-N ranking for a batch of users over a candidate list (WMF.rank,
// wmf_model.py:25-47).
//
// Round-1 design: the scores themselves are computed in the reference's exact fp32 rounding
// order (products rounded separately, NumPy pairwise reduce, biases added last), so the
// selected index set is the reference's by construction - no tensor-core candidate pass
// whose error would have to be bounded (SURVEY.md D6). One thread forms a whole dot product
// for 4 users at a time from a shared-memory tile of item rows (8 independent accumulators
// per user = NumPy's 8 strided partial sums, so the thread-serial order is the same order).
// Selection: per-user radix select on order-preserving keys + bitonic sort of the winners.
#include <stdlib.h>
#include "common.cuh"
#include "score.cuh"

namespace wmf {

constexpr int SC_THREADS = 128;  // items per tile (one per thread)
constexpr int SC_USERS = 32;     // users per CTA pass (8 groups of 4)
constexpr int TK_THREADS = 256;

// NumPy pairwise block (n <= 128) for 4 users sharing one item row; u rows are in smem.
__device__ __forceinline__ void np_block4(const float* __restrict__ u0, const float* __restrict__ u1,
                                          const float* __restrict__ u2, const float* __restrict__ u3,
                                          const float* __restrict__ v, int n, float out[4]) {
    const float* us[4] = {u0, u1, u2, u3};
    if (n < 8) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float acc = n > 0 ? __fmul_rn(us[q][0], v[0]) : 0.0f;
            for (int i = 1; i < n; ++i) acc = __fadd_rn(acc, __fmul_rn(us[q][i], v[i]));
            out[q] = acc;
        }
        return;
    }
    float r[4][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float vk = v[k];
#pragma unroll
        for (int q = 0; q < 4; ++q) r[q][k] = __fmul_rn(us[q][k], vk);
    }
    int i = 8;
    for (; i + 8 <= n; i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float vk = v[i + k];
#pragma unroll
            for (int q = 0; q < 4; ++q) r[q][k] = __fadd_rn(r[q][k], __fmul_rn(us[q][i + k], vk));
        }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float s = __fadd_rn(__fadd_rn(__fadd_rn(r[q][0], r[q][1]), __fadd_rn(r[q][2], r[q][3])),
                            __fadd_rn(__fadd_rn(r[q][4], r[q][5]), __fadd_rn(r[q][6], r[q][7])));
        for (int t = i; t < n; ++t) s = __fadd_rn(s, __fmul_rn(us[q][t], v[t]));
        out[q] = s;
    }
}

__device__ inline void np_dot4(const float* u0, const float* u1, const float* u2, const float* u3, const float* v,
                               int n, float out[4]) {
    if (n <= 128) { np_block4(u0, u1, u2, u3, v, n, out); return; }
    // two levels are enough for n <= 512 (WMF_MAX_F = 320)
    int segs[5];
    int half = n / 2; half -= half % 8;
    int nseg = 0;
    segs[0] = 0;
    auto push = [&](int off, int len) {
        if (len <= 128) { segs[++nseg] = off + len; }
        else { int h = len / 2; h -= h % 8; segs[++nseg] = off + h; segs[++nseg] = off + len; }
    };
    push(0, half);
    const int left_segs = nseg;
    push(half, n - half);
    float part[4][4];
    for (int s = 0; s < nseg; ++s) {
        float o[4];
        np_block4(u0 + segs[s], u1 + segs[s], u2 + segs[s], u3 + segs[s], v + segs[s], segs[s + 1] - segs[s], o);
#pragma unroll
        for (int q = 0; q < 4; ++q) part[s][q] = o[q];
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float a = left_segs == 2 ? __fadd_rn(part[0][q], part[1][q]) : part[0][q];
        float b = (nseg - left_segs) == 2 ? __fadd_rn(part[left_segs][q], part[left_segs + 1][q]) : part[left_segs][q];
        out[q] = __fadd_rn(a, b);
    }
}

// S[ub x ni] = exact scores of users[u0..u0+ub) against candidate items.
__global__ __launch_bounds__(SC_THREADS) void score_tile_kernel(const int64_t* __restrict__ users, int64_t u_begin,
                                                                int ub, const int64_t* __restrict__ cand, int64_t ni,
                                                                const float* __restrict__ U, int64_t ldu,
                                                                const float* __restrict__ V, int64_t ldv, int f,
                                                                int bias, float* __restrict__ S,
                                                                const int* __restrict__ run_if) {
    extern __shared__ __align__(16) float sm[];
    if (run_if != nullptr && *run_if == 0) return;  // fix-up launch after the tensor-core path: nothing overflowed
    const int FS = f + 1 + ((f & 1) ? 0 : 0);  // row stride (floats); f+1 keeps rows on distinct banks
    float* sV = sm;                            // SC_THREADS x FS
    float* sU = sm + (size_t)SC_THREADS * FS;  // SC_USERS x FS
    const int tid = threadIdx.x;
    const int64_t tiles_x = (ni + SC_THREADS - 1) / SC_THREADS, tiles_y = (ub + SC_USERS - 1) / SC_USERS;
    // grid-stride over (item tile, user tile): a conditional fix-up launch that has nothing to do exits cheaply
    for (int64_t tile = blockIdx.x; tile < tiles_x * tiles_y; tile += gridDim.x) {
    const int64_t i0 = (tile % tiles_x) * SC_THREADS;
    const int u_tile0 = (int)(tile / tiles_x) * SC_USERS;
    __syncthreads();  // the previous tile's shared-memory rows have been consumed
    // stage item rows (coalesced: consecutive threads read consecutive columns of one row)
    for (int r = 0; r < SC_THREADS; ++r) {
        const int64_t ip = i0 + r;
        const float* src = nullptr;
        if (ip < ni) src = V + (cand ? cand[ip] : ip) * ldv;
        for (int c = tid; c < f; c += SC_THREADS) sV[(size_t)r * FS + c] = src ? src[c] : 0.0f;
    }
    for (int r = 0; r < SC_USERS; ++r) {
        const int ul = u_tile0 + r;
        const float* src = nullptr;
        if (ul < ub) src = U + users[u_begin + ul] * ldu;
        for (int c = tid; c < f; c += SC_THREADS) sU[(size_t)r * FS + c] = src ? src[c] : 0.0f;
    }
    __syncthreads();
    const int64_t item_pos = i0 + tid;
    if (item_pos >= ni) continue;
    const float* v = sV + (size_t)tid * FS;
    const int off = bias ? 1 : 0;
    for (int g = 0; g < SC_USERS / 4; ++g) {
        const int ul = u_tile0 + g * 4;
        if (ul >= ub) break;
        const float* u0 = sU + (size_t)(g * 4 + 0) * FS;
        const float* u1 = sU + (size_t)(g * 4 + 1) * FS;
        const float* u2 = sU + (size_t)(g * 4 + 2) * FS;
        const float* u3 = sU + (size_t)(g * 4 + 3) * FS;
        float o[4];
        np_dot4(u0 + off, u1 + off, u2 + off, u3 + off, v + off, f - off, o);
        const float* us[4] = {u0, u1, u2, u3};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (ul + q < ub) {
                float s = o[q];
                if (bias) s = __fadd_rn(__fadd_rn(s, us[q][0]), v[0]);  // wmf_model.py:211
                S[(size_t)(ul + q) * ni + item_pos] = s;
            }
        }
    }
    }
}

// Excluded items of the users of a score tile: their scores become the all-ones bit pattern, which order_key maps
// to 0, below every other score. One CTA per user row (grid-stride).
template <typename T>
__global__ __launch_bounds__(256) void score_exclude_kernel(const int64_t* __restrict__ users, int64_t u_begin, int ub,
                                                            const int64_t* __restrict__ ex_indptr,
                                                            const int32_t* __restrict__ ex_indices, int64_t ni,
                                                            T* __restrict__ S, const int* __restrict__ run_if) {
    if (run_if != nullptr && *run_if == 0) return;
    for (int r = blockIdx.x; r < ub; r += gridDim.x) {
        const int64_t user = users[u_begin + r];
        const int64_t lo = ex_indptr[user], hi = ex_indptr[user + 1];
        for (int64_t e = lo + threadIdx.x; e < hi; e += blockDim.x)
            S[(size_t)r * ni + ex_indices[e]] = RankKey<T>::excluded();
    }
}

// One CTA per user row of S: k-th largest key by 8-bit radix select (4 passes for float, 8 for double), gather winners
// (ties at the threshold taken in candidate order), bitonic sort descending. `excl`: winners with key 0 are
// excluded items (score_exclude_kernel) a user with fewer than topn others is left with: id -1, score NaN.
template <typename T>
__global__ __launch_bounds__(TK_THREADS) void topk_rows_kernel(const T* __restrict__ S, int64_t ni, int topn,
                                                               const int64_t* __restrict__ cand,
                                                               int64_t* __restrict__ out_ids,
                                                               T* __restrict__ out_scores,
                                                               const int* __restrict__ run_if, int excl) {
    using R = RankKey<T>;
    using Key = typename R::Key;
    using Entry = typename R::Entry;
    __shared__ unsigned hist[256];
    if (run_if != nullptr && *run_if == 0) return;
    __shared__ Entry keys[TK_MAX];
    __shared__ Key s_prefix;
    __shared__ unsigned s_need, s_count, s_tie_base;
    __shared__ unsigned s_scan[TK_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const T* row = S + (size_t)blockIdx.x * ni;
    // --- radix select: find key T = topn-th largest
    Key prefix = 0, mask = 0;
    unsigned need = (unsigned)topn;
    for (int shift = R::BITS - 8; shift >= 0; shift -= 8) {
        hist[tid] = 0;
        __syncthreads();
        for (int64_t i = tid; i < ni; i += TK_THREADS) {
            const Key k = order_key(row[i]);
            if ((k & mask) == prefix) atomicAdd(&hist[(unsigned)(k >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid == 0) {
            unsigned acc = 0;
            int b = 255;
            for (; b > 0; --b) {
                if (acc + hist[b] >= need) break;
                acc += hist[b];
            }
            s_prefix = prefix | ((Key)b << shift);
            s_need = need - acc;  // how many still needed inside bucket b
        }
        __syncthreads();
        prefix = s_prefix;
        need = s_need;
        mask |= (Key)255u << shift;
        __syncthreads();
    }
    const Key T_ = prefix;           // threshold key
    const unsigned need_ties = need; // winners with key == T_, lowest positions first
    if (tid == 0) { s_count = 0; s_tie_base = 0; }
    __syncthreads();
    // --- strictly greater: any order (sorted afterwards)
    for (int64_t i = tid; i < ni; i += TK_THREADS) {
        const Key k = order_key(row[i]);
        if (k > T_) {
            unsigned slot = atomicAdd(&s_count, 1u);
            keys[slot] = R::entry(k, (uint32_t)i);
        }
    }
    __syncthreads();
    const unsigned n_gt = s_count;
    // --- ties in candidate order: ordered block scan over chunks of TK_THREADS
    for (int64_t base = 0; base < ni; base += TK_THREADS) {
        const unsigned taken = s_tie_base;
        if (taken >= need_ties) break;  // uniform (read after the barrier below / initial barrier)
        const int64_t i = base + tid;
        const bool is_tie = i < ni && order_key(row[i]) == T_;
        const unsigned bal = __ballot_sync(0xffffffffu, is_tie);
        if (lane == 0) s_scan[warp] = __popc(bal);
        __syncthreads();
        unsigned before = 0, total = 0;
        for (int w = 0; w < TK_THREADS / 32; ++w) {
            if (w < warp) before += s_scan[w];
            total += s_scan[w];
        }
        const unsigned rank = taken + before + __popc(bal & ((1u << lane) - 1u));
        if (is_tie && rank < need_ties) keys[n_gt + rank] = R::entry(T_, (uint32_t)i);
        __syncthreads();
        if (tid == 0) s_tie_base = taken + total;
        __syncthreads();
    }
    // --- bitonic sort (descending) of topn composite keys, padded to a power of two with key 0
    int npow = 1;
    while (npow < topn) npow <<= 1;
    for (int i = topn + tid; i < npow; i += TK_THREADS) keys[i] = R::entry(0, 0xFFFFFFFFu);
    __syncthreads();
    for (int size = 2; size <= npow; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < npow / 2; t += TK_THREADS) {
                const int lo = 2 * t - (t & (stride - 1));
                const int hi = lo + stride;
                const bool desc = ((lo & size) == 0);
                const Entry a = keys[lo], b = keys[hi];
                if (R::less(a, b) == desc) { keys[lo] = b; keys[hi] = a; }
            }
            __syncthreads();
        }
    }
    for (int t = tid; t < topn; t += TK_THREADS) {
        const Entry k = keys[t];
        const uint32_t pos = R::pos(k);
        const bool none = excl && R::key(k) == 0;
        out_ids[(size_t)blockIdx.x * topn + t] = none ? -1 : (cand ? cand[pos] : (int64_t)pos);
        if (out_scores) out_scores[(size_t)blockIdx.x * topn + t] = row[pos];
    }
}

int select_topk_double(const int64_t* users, int64_t u_begin, int ub, const int64_t* ex_indptr, const int32_t* ex_indices,
                       double* S, int64_t ni, int topn, int64_t* out_ids, double* out_scores, cudaStream_t st,
                       bool marked) {
    if (ex_indptr) {
        score_exclude_kernel<double><<<(unsigned)(ub < 65535 ? ub : 65535), 256, 0, st>>>(users, u_begin, ub, ex_indptr,
                                                                                           ex_indices, ni, S, nullptr);
        WMF_LAUNCH_CHECK("score_exclude_kernel<double>");
    }
    topk_rows_kernel<double><<<ub, TK_THREADS, 0, st>>>(S, ni, topn, nullptr, out_ids, out_scores, nullptr,
                                                        ex_indptr != nullptr || marked);
    WMF_LAUNCH_CHECK("topk_rows_kernel<double>");
    return WMF_OK;
}

static int64_t score_user_batch(int64_t nu, int64_t ni) {
    // keep the score tile near 64 MiB so the selection passes hit L2 (126 MB)
    int64_t ub = (64ll << 20) / (ni * 4 > 0 ? ni * 4 : 4);
    if (ub < SC_USERS) ub = SC_USERS;
    ub = ub / SC_USERS * SC_USERS;
    if (ub > 65535ll * SC_USERS) ub = 65535ll * SC_USERS;
    if (ub > nu) ub = nu;
    return ub;
}

}  // namespace wmf

using namespace wmf;

extern "C" {

size_t wmf_score_topk_workspace_bytes(int64_t nu, int64_t ni, int topn) {
    (void)topn;
    if (nu <= 0 || ni <= 0) return 0;
    const size_t exact = align_up((size_t)score_user_batch(nu, ni) * (size_t)ni * sizeof(float), 1024);
    const size_t tc = exact + score_tc_workspace_bytes(nu, ni);  // the query does not know f: assume the tensor-core path
    return exact > tc ? exact : tc;
}

size_t wmf_score_topk_exclude_workspace_bytes(int64_t nu, int64_t ni, int topn) {
    return wmf_score_topk_workspace_bytes(nu, ni, topn);
}

}  // extern "C"

// wmf_score_topk, and wmf_score_topk_exclude when ex_indptr is not null
static int score_topk(const char* name, const int64_t* users, int64_t nu, const int64_t* cand,
                      const int64_t* ex_indptr, const int32_t* ex_indices, int64_t ni, const float* U, int64_t ldu,
                      const float* V, int64_t ldv, int f, int bias, int topn, int64_t* out_ids, float* out_scores,
                      int32_t* fixup_users, void* ws, size_t ws_bytes, void* stream) {
    WMF_REQUIRE(f > 0 && f <= WMF_MAX_F && (!bias || f >= 2), "%s: f=%d out of range", name, f);
    WMF_REQUIRE(nu >= 0 && ni >= 0, "%s: negative size", name);
    cudaStream_t st = (cudaStream_t)stream;
    if (fixup_users) WMF_CUDA(cudaMemsetAsync(fixup_users, 0, sizeof(int32_t), st));
    if (nu == 0 || topn == 0) return WMF_OK;
    WMF_REQUIRE(users && U && V && out_ids, "%s: null argument", name);
    WMF_REQUIRE(ni < (1ll << 32), "%s: more than 2^32 candidates", name);
    if (topn < 0 || topn > ni || topn > TK_MAX) {
        set_error("%s: topn=%d outside 1..min(ni=%lld, %d)", name, topn, (long long)ni, TK_MAX);
        return WMF_ERR_UNSUPPORTED;
    }
    size_t need = wmf_score_topk_workspace_bytes(nu, ni, topn);
    if (ws == nullptr || ws_bytes < need) {
        set_error("%s: workspace %zu < %zu", name, ws_bytes, need);
        return WMF_ERR_WORKSPACE;
    }
    const int FS = f + 1;
    const size_t smem = (size_t)(SC_THREADS + SC_USERS) * FS * sizeof(float);
    WMF_CUDA(cudaFuncSetAttribute(score_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t ubatch = score_user_batch(nu, ni);
    float* S = (float*)ws;
    const size_t exact_bytes = align_up((size_t)ubatch * (size_t)ni * sizeof(float), 1024);
    // Tensor-core candidate generation + exact rescoring when the shape allows it (WMF_SCORE_EXACT=1 forces
    // the exact CUDA-core kernels); afterwards the exact kernels run only if a user overflowed its candidate list.
    const bool use_tc = score_tc_supported(ni, f, bias, topn) && getenv("WMF_SCORE_EXACT") == nullptr &&
                        ws_bytes >= exact_bytes + score_tc_workspace_bytes(nu, ni);
    int* redo = nullptr;
    if (use_tc) {
        const int64_t tb = score_tc_user_batch(nu);
        for (int64_t u0 = 0; u0 < nu; u0 += tb) {
            const int ub = (int)((nu - u0) < tb ? (nu - u0) : tb);
            int rc = score_topk_tc_batch(users, u0, ub, tb, cand, ni, U, ldu, V, ldv, f, bias, topn, out_ids, out_scores,
                                         (char*)ws + exact_bytes, u0 == 0, &redo, st, ex_indptr, ex_indices, fixup_users);
            if (rc) return rc;
        }
    }
    int64_t xbatch = ubatch;
    if (use_tc) {  // conditional fix-up after the tensor-core path: few large batches in its dead scratch regions
        size_t off = 0, bytes = 0;
        score_tc_fixup_region(nu, ni, &off, &bytes);
        int64_t xb = (int64_t)(bytes / ((size_t)ni * sizeof(float))) / SC_USERS * SC_USERS;
        if (xb > 65535ll * SC_USERS) xb = 65535ll * SC_USERS;
        if (xb > ubatch) { xbatch = xb; S = (float*)((char*)ws + exact_bytes + off); }
    }
    for (int64_t u0 = 0; u0 < nu; u0 += xbatch) {
        const int ub = (int)((nu - u0) < xbatch ? (nu - u0) : xbatch);
        const int64_t tiles = ((ni + SC_THREADS - 1) / SC_THREADS) * ((ub + SC_USERS - 1) / SC_USERS);
        const int64_t cap = (int64_t)sm_count() * 8;
        const unsigned grid = (unsigned)(tiles < cap ? tiles : cap);
        score_tile_kernel<<<grid, SC_THREADS, smem, st>>>(users, u0, ub, cand, ni, U, ldu, V, ldv, f, bias, S, redo);
        WMF_LAUNCH_CHECK("score_tile_kernel");
        if (ex_indptr) {
            score_exclude_kernel<<<(unsigned)(ub < 65535 ? ub : 65535), 256, 0, st>>>(users, u0, ub, ex_indptr, ex_indices,
                                                                                      ni, S, redo);
            WMF_LAUNCH_CHECK("score_exclude_kernel");
        }
        topk_rows_kernel<<<ub, TK_THREADS, 0, st>>>(S, ni, topn, cand, out_ids + (size_t)u0 * topn,
                                                    out_scores ? out_scores + (size_t)u0 * topn : nullptr, redo,
                                                    ex_indptr != nullptr);
        WMF_LAUNCH_CHECK("topk_rows_kernel");
    }
    return WMF_OK;
}

extern "C" {

int wmf_score_topk(const int64_t* users, int64_t nu, const int64_t* cand, int64_t ni, const float* U, int64_t ldu,
                   const float* V, int64_t ldv, int f, int bias, int topn, int64_t* out_ids, float* out_scores,
                   void* ws, size_t ws_bytes, void* stream) {
    return score_topk("wmf_score_topk", users, nu, cand, nullptr, nullptr, ni, U, ldu, V, ldv, f, bias, topn, out_ids,
                      out_scores, nullptr, ws, ws_bytes, stream);
}

int wmf_score_topk_exclude(const int64_t* users, int64_t nu, const int64_t* ex_indptr, const int32_t* ex_indices,
                           int64_t ni, const float* U, int64_t ldu, const float* V, int64_t ldv, int f, int bias,
                           int topn, int64_t* out_ids, float* out_scores, int32_t* fixup_users, void* ws,
                           size_t ws_bytes, void* stream) {
    WMF_REQUIRE(ex_indptr, "wmf_score_topk_exclude: null exclusion matrix");  // ex_indices may be null when it is empty
    return score_topk("wmf_score_topk_exclude", users, nu, nullptr, ex_indptr, ex_indices, ni, U, ldu, V, ldv, f, bias,
                      topn, out_ids, out_scores, fixup_users, ws, ws_bytes, stream);
}

}  // extern "C"
