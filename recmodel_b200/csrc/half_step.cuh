// Parameter block and internal entry points shared by the half-step implementations.
#pragma once
#include "common.cuh"

namespace wmf {

struct HalfStepParams {
    const int64_t* indptr;
    const int32_t* indices;
    const float* data;
    int64_t rows;
    const int32_t* row_order;
    int64_t sched_len;  // schedule slots to walk: order_len, or rows without a schedule
    const float* Y;
    int64_t ldy;
    int f;
    const float* G;
    int bias;
    float* X;
    int64_t ldx;
    int64_t cols;       // rows of Y (= columns of the count matrix); the tcgen05 path whitens all of them
    // filled by the implementation
    int* counter;
    long long* prof;    // nullable: per-role cycle counters of CTA 0 (tcgen05 kernels, profiling builds)
    const int* run_if;  // nullable: the SIMT kernel returns at once when *run_if == 0
    const int* sched_len_dev;  // nullable: the SIMT kernel walks *sched_len_dev slots (device-side fix-up list)
    float* slab;
    int lda;
    int FP;
    int KC;
    // tcgen05 path: Y / X above are the whitened factors and the whitened solution (ld = FP)
    const float* Yraw;  // original factors: column 0 holds the bias the weights are shifted by (wmf_model.py:343)
    int64_t ldraw;
    int f8, f16;        // f rounded up to 8 / 16: Gauss-Jordan steps and MMA widths stop there
    int* fix_list;      // rows the CUDA-core LU kernel solves afterwards (negative weights, failed pivot)
    int* fix_count;
    int nd_max;         // rows with at most this many entries take the dual (n x n) kernel
    int cg_maxit;       // matrix-vector products the conjugate-gradient solver may spend on a row before the in-TMEM
                        // factorisation takes it; 0: factorisation only (WMF_ALGO_TCGEN05_DIRECT)
};

size_t simt_half_step_workspace_bytes(int f);
int simt_half_step(const HalfStepParams& in, void* ws, size_t ws_bytes, cudaStream_t st);
bool tc_half_step_supported(int f, int bias);
size_t tc_half_step_workspace_bytes(int64_t rows, int64_t cols, int f, int bias, int64_t segments);  // segments < 0: default scratch
int tc_half_step(const HalfStepParams& in, void* ws, size_t ws_bytes, cudaStream_t st);
// dual (n x n) kernel for the packs of short rows of the pack table (half_step_dual.cu)
int tc_dual_launch(const HalfStepParams& p, const int4* ptab, const uint32_t* hdr_u, int grid, cudaStream_t st);
int tc_dual_max_entries();
int tc_cg_max_products();   // default budget of the conjugate-gradient solver (WMF_TC_CG=<n> overrides, 0 = off)
// primal kernel for 128 < f <= 256 (half_step_tc256.cu); same tables and scratch conventions as the 128-wide one
size_t tc256_part_floats();
int tc256_launch(const HalfStepParams& p, const int4* tab, const int4* segtab, float* parts, int* counters,
                 const uint32_t* hdr_u, int64_t extra_slot0, int* flags, int grid, cudaStream_t st);

}  // namespace wmf
