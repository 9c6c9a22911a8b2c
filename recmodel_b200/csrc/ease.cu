// N4 (SURVEY.md 8f): the EASE model of the reference (RecModel/ease_model.py:81-114), the WMF path's closest sibling:
// one dense item x item Gram and one dense inverse instead of many small ones.
//   G = X^T X + alpha I                      ease_model.py:93,97   -> ease_gram_kernel (one warp per user row)
//   P = inv(G)                               :102                  -> blocked in-place Gauss-Jordan (no pivoting: G is SPD)
//   W = P / (-diag(P) + 1e-9), diag(W) = 0   :106-108              -> ease_finish_kernel
//   predict: sum_j X[u, j] W[j, item]        fast_utils/ease_utils.pyx:15-30 -> ease_predict_kernel
//   top-N of a user's unseen items (Ease.recommend)                 -> ease_score_tile_kernel + the exact selection
// The inverse is n^3 FP32 FMAs as rank-64 updates (register-blocked 128 x 128 tiles): compute-bound on the CUDA
// cores, 0.6 s at the 26 744 items of ML-20M; the reference does the same arithmetic in FP32 LAPACK (sgetri).
#include "common.cuh"
#include "score.cuh"

namespace wmf {

namespace {

constexpr int ENB = 64;   // panel width of the blocked inverse

// G[a][b] += x_a x_b over the pairs of one user's stored entries (G pre-filled with alpha on the diagonal).
// Counts are small integers, so the FP32 atomic sums are exact whatever their order.
__global__ void ease_gram_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                 const float* __restrict__ data, int64_t rows, int64_t n, float* __restrict__ G) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= rows) return;
    const int lane = threadIdx.x & 31;
    const int64_t lo = indptr[r], hi = indptr[r + 1];
    for (int64_t a = lo; a < hi; ++a) {
        const float xa = data[a];
        float* grow = G + (int64_t)indices[a] * n;
        for (int64_t b = lo + lane; b < hi; b += 32) atomicAdd(grow + indices[b], xa * data[b]);
    }
}

__global__ void ease_fill_diag_kernel(float* __restrict__ G, int64_t n, float alpha) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) G[i * n + i] = alpha;
}

// Dinv = inverse of the ENB x ENB diagonal block (Gauss-Jordan without pivoting, one CTA, shared memory)
__global__ void __launch_bounds__(256) ease_diag_inverse_kernel(const float* __restrict__ A, int64_t n, int64_t k0, int nb,
                                                                float* __restrict__ Dinv, int* __restrict__ flag) {
    __shared__ float M[ENB][2 * ENB + 1];
    const int tid = threadIdx.x;
    for (int e = tid; e < nb * nb; e += 256) {
        const int i = e / nb, j = e % nb;
        M[i][j] = A[(k0 + i) * n + k0 + j];
        M[i][nb + j] = i == j ? 1.0f : 0.0f;
    }
    __syncthreads();
    for (int k = 0; k < nb; ++k) {
        const float piv = M[k][k];
        __syncthreads();
        if (tid == 0 && !(fabsf(piv) > 0.0f)) atomicOr(flag, 1);
        const float inv = 1.0f / piv;
        for (int j = tid; j < 2 * nb; j += 256) M[k][j] *= inv;
        __syncthreads();
        for (int e = tid; e < nb * 2 * nb; e += 256) {
            const int i = e / (2 * nb), j = e % (2 * nb);
            if (i != k && j != k) M[i][j] = fmaf(-M[i][k], M[k][j], M[i][j]);
        }
        __syncthreads();
        for (int i = tid; i < nb; i += 256) if (i != k) M[i][k] = 0.0f;
        __syncthreads();
    }
    for (int e = tid; e < nb * nb; e += 256) Dinv[e] = M[e / nb][nb + e % nb];
}

// Panel step k of the in-place block Gauss-Jordan inversion:
//   C = A[:, K] (saved, n x nb);  R = Dinv A[K, :] with R[:, K] = Dinv (nb x n);  then (update kernel) for rows outside K:
//   A[i, :] = (j in K ? 0 : A[i, :]) - C[i, :] R,  and A[K, :] = R.
__global__ void ease_panel_kernel(float* __restrict__ A, int64_t n, int64_t k0, int nb, const float* __restrict__ Dinv,
                                  float* __restrict__ C, float* __restrict__ R) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // column (for R) / row (for C)
    if (j >= n) return;
    float col[ENB];
    for (int c = 0; c < nb; ++c) {
        C[j * ENB + c] = A[j * n + k0 + c];        // row j of the column panel
        col[c] = A[(k0 + c) * n + j];              // column j of the row panel
    }
    const bool inK = j >= k0 && j < k0 + nb;
    for (int r = 0; r < nb; ++r) {
        float acc = 0.0f;
        if (inK) acc = Dinv[r * nb + (j - k0)];
        else for (int c = 0; c < nb; ++c) acc = fmaf(Dinv[r * nb + c], col[c], acc);
        R[(int64_t)r * n + j] = acc;
    }
}

// A[i][j] = (i in K ? R[i-k0][j] : (j in K ? 0 : A[i][j]) - sum_c C[i][c] R[c][j]); 128 x 128 tiles, 8 x 8 per thread
__global__ void __launch_bounds__(256) ease_update_kernel(float* __restrict__ A, int64_t n, int64_t k0, int nb,
                                                          const float* __restrict__ C, const float* __restrict__ R) {
    constexpr int KC = 32;                            // the rank-64 update in two chunks of 32 (48 KB of static shared memory)
    __shared__ __align__(16) float Cs[KC][128 + 4];   // [c][row]
    __shared__ __align__(16) float Rs[KC][128];       // [c][col]
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int64_t i0 = (int64_t)blockIdx.y * 128, j0 = (int64_t)blockIdx.x * 128;
    float acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.0f;
    for (int c0 = 0; c0 < ENB; c0 += KC) {
        __syncthreads();
        for (int e = tid; e < 128 * KC; e += 256) {
            const int r = e / KC, c = e % KC;
            Cs[c][r] = (i0 + r < n && c0 + c < nb) ? C[(i0 + r) * ENB + c0 + c] : 0.0f;
        }
        for (int e = tid; e < KC * 128; e += 256) {
            const int c = e / 128, jj = e % 128;
            Rs[c][jj] = (j0 + jj < n && c0 + c < nb) ? R[(int64_t)(c0 + c) * n + j0 + jj] : 0.0f;
        }
        __syncthreads();
#pragma unroll 8
        for (int c = 0; c < KC; ++c) {
            const float4 a0 = *reinterpret_cast<const float4*>(&Cs[c][ty * 8]), a1 = *reinterpret_cast<const float4*>(&Cs[c][ty * 8 + 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Rs[c][tx * 8]), b1 = *reinterpret_cast<const float4*>(&Rs[c][tx * 8 + 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(av[a], bv[b], acc[a][b]);
        }
    }
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        const int64_t i = i0 + ty * 8 + a;
        if (i >= n) continue;
        const bool rowK = i >= k0 && i < k0 + nb;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int64_t j = j0 + tx * 8 + b;
            if (j >= n) continue;
            float v;
            if (rowK) v = R[(int64_t)(i - k0) * n + j];
            else {
                const bool colK = j >= k0 && j < k0 + nb;
                v = (colK ? 0.0f : A[i * n + j]) - acc[a][b];
            }
            A[i * n + j] = v;
        }
    }
}

// W = P / (-diag(P) + 1e-9) column-wise, then a zero diagonal (ease_model.py:106-108)
__global__ void ease_finish_kernel(float* __restrict__ P, int64_t n, const float* __restrict__ diag) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * n) return;
    const int64_t i = e / n, j = e % n;
    P[e] = i == j ? 0.0f : P[e] / (-diag[j] + 1e-9f);
}
__global__ void ease_diag_kernel(const float* __restrict__ P, int64_t n, float* __restrict__ diag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) diag[i] = P[i * n + i];
}

// out[k] = sum_j X[u_k, j] W[j, item_k]: FP32 products summed in double in stored order, as the reference's loop does
__global__ void ease_predict_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                    const float* __restrict__ data, const float* __restrict__ W, int64_t n,
                                    const int64_t* __restrict__ users, int64_t user_stride, const int64_t* __restrict__ items,
                                    int64_t count, double* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const int64_t u = users[k * user_stride], it = items[k];
    double acc = 0.0;
    for (int64_t j = indptr[u]; j < indptr[u + 1]; ++j) acc += (double)__fmul_rn(data[j], W[(int64_t)indices[j] * n + it]);
    out[k] = acc;
}

constexpr int ES_THREADS = 128;  // item columns per CTA (one per thread)
constexpr int ES_USERS = 4;      // users per CTA

// S[r][i] = sum_j X[users[u_begin + r], j] W[j, i] for the ub users of a batch, with the arithmetic of
// ease_predict_kernel (so every score is bitwise what wmf_ease_predict returns). CTA = (item panel, group of ES_USERS
// users); the item panel is the outer index, so the CTAs running together share a panel of W, which is fetched from
// HBM about once per batch and read from L2 by the other users of the batch.
__global__ __launch_bounds__(ES_THREADS) void ease_score_tile_kernel(const int64_t* __restrict__ indptr,
                                                                     const int32_t* __restrict__ indices,
                                                                     const float* __restrict__ data,
                                                                     const float* __restrict__ W, int64_t n,
                                                                     const int64_t* __restrict__ users, int64_t u_begin,
                                                                     int ub, double* __restrict__ S) {
    const int groups = (ub + ES_USERS - 1) / ES_USERS;
    const int64_t panel = blockIdx.x / groups;
    const int g = (int)(blockIdx.x % groups);
    const int64_t i = panel * ES_THREADS + threadIdx.x;
    if (i >= n) return;
    const float* __restrict__ Wi = W + i;
    for (int q = 0; q < ES_USERS; ++q) {
        const int r = g * ES_USERS + q;
        if (r >= ub) break;
        const int64_t u = users[u_begin + r];
        const int64_t lo = indptr[u], hi = indptr[u + 1];
        double acc = 0.0;
        int64_t e = lo;
        for (; e + 4 <= hi; e += 4) {  // loads first, then the adds in stored order
            const float w0 = Wi[(int64_t)indices[e] * n], w1 = Wi[(int64_t)indices[e + 1] * n];
            const float w2 = Wi[(int64_t)indices[e + 2] * n], w3 = Wi[(int64_t)indices[e + 3] * n];
            acc += (double)__fmul_rn(data[e], w0);
            acc += (double)__fmul_rn(data[e + 1], w1);
            acc += (double)__fmul_rn(data[e + 2], w2);
            acc += (double)__fmul_rn(data[e + 3], w3);
        }
        for (; e < hi; ++e) acc += (double)__fmul_rn(data[e], Wi[(int64_t)indices[e] * n]);
        S[(size_t)r * n + i] = acc;
    }
}

// users per score tile: keep the [ub x n] double tile near 64 MiB so the selection passes hit L2 (126 MB)
int64_t ease_user_batch(int64_t nu, int64_t n) {
    int64_t ub = (64ll << 20) / (n * 8);
    if (ub < ES_USERS) ub = ES_USERS;
    ub = ub / ES_USERS * ES_USERS;
    if (ub > nu) ub = nu;
    return ub;
}

}  // namespace

}  // namespace wmf

using namespace wmf;

extern "C" {

size_t wmf_ease_workspace_bytes(int64_t n) {   // Dinv, column panel C, row panel R, diagonal, flag
    return align_up((size_t)ENB * ENB * 4, 256) + align_up((size_t)n * ENB * 4, 256) * 2 + align_up((size_t)n * 4, 256) + 256;
}

int wmf_ease_train(const int64_t* indptr, const int32_t* indices, const float* data, int64_t rows, int64_t n, float alpha,
                   float* W, void* ws, size_t ws_bytes, void* stream) {
    WMF_REQUIRE(indptr && W && rows >= 0 && n > 0 && n < (1ll << 31), "wmf_ease_train: bad arguments");
    WMF_REQUIRE(ws && ws_bytes >= wmf_ease_workspace_bytes(n), "wmf_ease_train: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    char* base = reinterpret_cast<char*>(ws);
    float* Dinv = reinterpret_cast<float*>(base);
    float* C = reinterpret_cast<float*>(base + align_up((size_t)ENB * ENB * 4, 256));
    float* R = C + align_up((size_t)n * ENB * 4, 256) / 4;
    float* diag = R + align_up((size_t)n * ENB * 4, 256) / 4;
    int* flag = reinterpret_cast<int*>(reinterpret_cast<char*>(diag) + align_up((size_t)n * 4, 256));
    WMF_CUDA(cudaMemsetAsync(W, 0, (size_t)n * n * 4, st));
    WMF_CUDA(cudaMemsetAsync(flag, 0, 4, st));
    ease_fill_diag_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(W, n, alpha);
    WMF_LAUNCH_CHECK("ease_fill_diag_kernel");
    if (rows > 0) {
        ease_gram_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(indptr, indices, data, rows, n, W);
        WMF_LAUNCH_CHECK("ease_gram_kernel");
    }
    const unsigned tiles = (unsigned)((n + 127) / 128);
    for (int64_t k0 = 0; k0 < n; k0 += ENB) {
        const int nb = (int)(n - k0 < ENB ? n - k0 : ENB);
        ease_diag_inverse_kernel<<<1, 256, 0, st>>>(W, n, k0, nb, Dinv, flag);
        WMF_LAUNCH_CHECK("ease_diag_inverse_kernel");
        ease_panel_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(W, n, k0, nb, Dinv, C, R);
        WMF_LAUNCH_CHECK("ease_panel_kernel");
        ease_update_kernel<<<dim3(tiles, tiles), 256, 0, st>>>(W, n, k0, nb, C, R);
        WMF_LAUNCH_CHECK("ease_update_kernel");
    }
    ease_diag_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(W, n, diag);
    WMF_LAUNCH_CHECK("ease_diag_kernel");
    ease_finish_kernel<<<(unsigned)(((size_t)n * n + 255) / 256), 256, 0, st>>>(W, n, diag);
    WMF_LAUNCH_CHECK("ease_finish_kernel");
    return WMF_OK;
}

int wmf_ease_predict(const int64_t* indptr, const int32_t* indices, const float* data, const float* W, int64_t n,
                     const int64_t* users, int64_t user_stride, const int64_t* items, int64_t count, double* out, void* stream) {
    WMF_REQUIRE(indptr && W && users && items && out && count >= 0, "wmf_ease_predict: bad arguments");
    if (count == 0) return WMF_OK;
    ease_predict_kernel<<<(unsigned)((count + 127) / 128), 128, 0, (cudaStream_t)stream>>>(indptr, indices, data, W, n, users,
                                                                                      user_stride, items, count, out);
    WMF_LAUNCH_CHECK("ease_predict_kernel");
    return WMF_OK;
}

size_t wmf_ease_score_topk_workspace_bytes(int64_t nu, int64_t n, int topn) {
    (void)topn;
    return score_topk_double_workspace_bytes(nu, n, ease_user_batch);
}

int wmf_ease_score_topk(const int64_t* x_indptr, const int32_t* x_indices, const float* x_data, const float* W,
                        int64_t n, const int64_t* users, int64_t nu, const int64_t* ex_indptr,
                        const int32_t* ex_indices, int topn, int64_t* out_ids, double* out_scores, void* ws,
                        size_t ws_bytes, void* stream) {
    return score_topk_double("wmf_ease_score_topk", x_indptr && W, ease_user_batch, n, users, nu, ex_indptr, ex_indices,
                             topn, out_ids, out_scores, ws, ws_bytes, stream,
                             [&](int64_t u0, int ub, double* S, cudaStream_t st) {
        const int64_t grid = (n + ES_THREADS - 1) / ES_THREADS * ((ub + ES_USERS - 1) / ES_USERS);
        ease_score_tile_kernel<<<(unsigned)grid, ES_THREADS, 0, st>>>(x_indptr, x_indices, x_data, W, n, users, u0, ub, S);
        WMF_LAUNCH_CHECK("ease_score_tile_kernel");
        return WMF_OK;
    });
}

}  // extern "C"
