// Shared by the exact (score.cu) and tensor-core (score_tc.cu) ranking paths.
#pragma once
#include "common.cuh"

namespace wmf {

// order-preserving map float -> uint32 (larger float -> larger key)
__device__ __forceinline__ uint32_t order_key(float x) {
    uint32_t b = __float_as_uint(x);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
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
