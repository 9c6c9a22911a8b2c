// K4 + K5 (tensor-core version): top-N ranking for a batch of users (WMF.rank, wmf_model.py:25-47).
//
// SURVEY.md D6: a tensor-core GEMM cannot reproduce NumPy's rounding order, so it cannot decide the
// top-N set by itself. It can decide which items CANNOT be in it:
//
//   K4  S~ = U~ V~^T on tcgen05 (kind::f16, fp32 accumulation in TMEM). U~, V~ are the factor rows
//       (with the bias columns folded in as two extra features), scaled by a power of two per matrix and
//       rounded to FP16. Operand tiles are written once by a prep kernel as ready-made 128-byte-swizzled
//       K-major images, so a tile reaches shared memory with ONE bulk-copy (TMA, UBLKCP) instruction.
//       |S~_ui / (su sv) - s_ui| <= eps_ui = c * ||u~|| * ||v~_i|| / (su sv) + delta for the exact NumPy-order
//       score s_ui, c = 1.02 * 2^-10 (two 11-bit roundings per product, fp32 accumulation, NumPy's own
//       rounding), delta covers FP16 subnormals.
//   K5  fused selection, nothing of S~ is written to memory. The GEMM runs twice over the same operands:
//       pass 1 keeps, per user, the maximum of every 32-item column block (from the accumulator in TMEM);
//       tau' = N-th largest block maximum is a lower bound of the N-th largest S~ (N distinct items reach
//       it). Every item of the exact top-N has S~ >= tau - 2 eps_u >= tau' - 2 eps_u (eps_u = max_i eps_ui):
//       with N items at S~ >= tau the exact N-th score t* is >= tau - eps, and an item with exact score
//       >= t* has S~ >= t* - eps. Pass 2 recomputes the tiles and appends the items above that threshold to
//       a per-user candidate list (about N + 10 at ML-20M shape); the candidates are rescored in the exact
//       NumPy order and the final top-N is selected from them, ties by candidate position: the same index
//       set and order as the exact path. If a user collects more than 1024 candidates (e.g. all scores
//       equal) a flag makes the caller redo the call with the exact CUDA-core kernels.
//   Exclusion (wmf_score_topk_exclude, EXCL = true): every epilogue thread walks its user's sorted list of
//       excluded item ids with one cursor, in step with the ascending 32-column blocks, and turns the ids that
//       fall into the block into a 32-bit mask. Pass 1 leaves masked columns out of the block maximum (a block
//       with nothing left gives -3e38), so tau' is still reached by N distinct items that may be returned and
//       the bound above holds for the top-N over the unseen items; pass 2 drops masked columns from the hits.
//       A user with fewer than N unseen items has -3e38 as its N-th block maximum: the threshold admits every
//       unseen item, the list is complete, and the rescoring pads it with id -1 instead of raising the flag.
#include <climits>
#include <cuda_fp16.h>
#include "common.cuh"
#include "score.cuh"

namespace wmf {
namespace stc {

constexpr int K = 128;                    // padded feature count of the tensor-core pass
constexpr int TM = 128, TN = 128;         // users x items per accumulator tile
constexpr int TILE_BYTES = TM * K * 2;    // 32 KB: two K-halves, each 128 rows x 128 B, 128-byte swizzled
constexpr int NB_STAGE = 3;               // item-tile stages
constexpr int OFF_A = 0;
constexpr int OFF_B = OFF_A + TILE_BYTES;
constexpr int OFF_BARS = OFF_B + NB_STAGE * TILE_BYTES;
constexpr int NBARS = 1 + 2 * NB_STAGE + 4;
constexpr int OFF_TMEM = OFF_BARS + NBARS * 8;
constexpr int SMEM_BYTES = OFF_TMEM + 16 + 1024;
constexpr int GEMM_THREADS = 192;         // warps 0-3 epilogue, warp 4 bulk-copy producer, warp 5 MMA issue
constexpr int CAND_MAX = 1024;            // candidate list capacity per user
constexpr int SUB = 32;                   // column block of the pass-1 maxima
constexpr int MAXSUB = 8192;              // most column blocks the threshold kernel takes (262 144 items)
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(bar), "r"(parity), "r"(0x989680u) : "memory");
}
// TMA bulk copy (linear): global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// K-major, 128-byte swizzle, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
           (2ull << 61);
}
constexpr uint32_t IDESC_F16_M128_N128 = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------
// prep: absolute maximum of the selected rows, then FP16 tile images + row norms
// ---------------------------------------------------------------------------------------------------
__global__ void stc_absmax_kernel(const int64_t* __restrict__ ids, int64_t id0, int64_t n, const float* __restrict__ X,
                                  int64_t ld, int f, uint32_t* __restrict__ out) {
    float m = 0.0f;
    const int64_t total = n * f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / f;
        const int c = (int)(i - r * f);
        const int64_t row = ids ? ids[id0 + r] : id0 + r;
        m = fmaxf(m, fabsf(X[row * ld + c]));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.0f) atomicMax(out, __float_as_uint(m));
}

__device__ __forceinline__ float pow2_scale(float absmax, int bias) {
    float m = bias ? fmaxf(absmax, 1.0f) : absmax;  // the folded bias columns hold the constant 1
    if (!(m > 0.0f) || !(m < 3.0e38f)) return 1.0f;
    int e = (int)floorf(log2f(16384.0f / m));
    if (ldexpf(m, e) >= 16384.0f) --e;  // scaled maximum in [2^13, 2^14)
    e = e > 60 ? 60 : (e < -60 ? -60 : e);
    return exp2f((float)e);
}

// One warp per (padded) row: lane l converts features 4l .. 4l+3. side 0 = users ([b, 1, x1..]), side 1 =
// items ([1, b, x1..]) when the bias columns are folded in. Rows >= n are zero (padding of the last tile).
__global__ void stc_convert_kernel(const int64_t* __restrict__ ids, int64_t id0, int64_t n, int64_t n_pad,
                                   const float* __restrict__ X, int64_t ld, int f, int bias, int side,
                                   const uint32_t* __restrict__ absmax, uint8_t* __restrict__ tiles,
                                   float* __restrict__ norms) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= n_pad) return;
    const float s = pow2_scale(__uint_as_float(*absmax), bias);
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < n) {
        const float* src = X + (ids ? ids[id0 + r] : id0 + r) * ld;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = 4 * lane + j;
            float x = 0.0f;
            if (!bias) {
                if (k < f) x = src[k];
            } else {
                if (k == 0) x = side == 0 ? src[0] : 1.0f;
                else if (k == 1) x = side == 0 ? 1.0f : src[0];
                else if (k <= f) x = src[k - 1];
            }
            v[j] = x * s;
        }
    }
    float nn = v[0] * v[0] + v[1] * v[1] + v[2] * v[2] + v[3] * v[3];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nn += __shfl_xor_sync(0xffffffffu, nn, o);
    if (lane == 0) norms[r] = sqrtf(nn) * 1.000001f;
    const __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
    const int64_t tile = r >> 7;
    const int rr = (int)(r & 127), k0 = 4 * lane, khalf = k0 >> 6, kk = k0 & 63;
    uint8_t* dst = tiles + tile * TILE_BYTES + khalf * (TILE_BYTES / 2) + rr * 128 + (((kk >> 3) ^ (rr & 7)) << 4) +
                   (kk & 7) * 2;
    *reinterpret_cast<uint2*>(dst) = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
}

// vmax[0] = max_i norms[i]
__global__ void stc_maxnorm_kernel(const float* __restrict__ norms, int64_t n, uint32_t* __restrict__ out) {
    float m = 0.0f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        m = fmaxf(m, norms[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.0f) atomicMax(out, __float_as_uint(m));
}

// ---------------------------------------------------------------------------------------------------
// K4: S~ = U~ V~^T tile by tile, one CTA per 128 users, item tiles streamed by bulk copies.
// MODE 0: per user maxima of every 32-column block.  MODE 1: append the items with S~ >= thr[user].
// EXCL: the item ids ex_indices[ex_indptr[user] ..) (ascending) of user = users[u_begin + row] take no part.
// ---------------------------------------------------------------------------------------------------
template <int MODE, bool EXCL>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
stc_gemm_kernel(const uint8_t* __restrict__ a_tiles, const uint8_t* __restrict__ b_tiles, int n_item_tiles, int ub,
                int64_t ni, float* __restrict__ maxima, const float* __restrict__ thr, int* __restrict__ cnt,
                uint32_t* __restrict__ lists, const int64_t* __restrict__ users, int64_t u_begin,
                const int64_t* __restrict__ ex_indptr, const int32_t* __restrict__ ex_indices) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = base + OFF_BARS;
    auto bar_a = [&]() { return bars; };
    auto bar_bfull = [&](int s) { return bars + 8u * (1 + s); };
    auto bar_bempty = [&](int s) { return bars + 8u * (1 + NB_STAGE + s); };
    auto bar_accfull = [&](int a) { return bars + 8u * (1 + 2 * NB_STAGE + a); };
    auto bar_accempty = [&](int a) { return bars + 8u * (1 + 2 * NB_STAGE + 2 + a); };
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        mbar_init(bar_a(), 1);
        for (int s = 0; s < NB_STAGE; ++s) { mbar_init(bar_bfull(s), 1); mbar_init(bar_bempty(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_accfull(a), 1); mbar_init(bar_accempty(a), 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(base + OFF_TMEM) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(base + OFF_TMEM));
    const int64_t u0 = (int64_t)blockIdx.x * TM;

    if (warp == 4) {
        if (lane == 0) {  // producer: one bulk copy per tile image
            mbar_expect_tx(bar_a(), TILE_BYTES);
            bulk_g2s(base + OFF_A, a_tiles + (int64_t)blockIdx.x * TILE_BYTES, TILE_BYTES, bar_a());
            for (int it = 0; it < n_item_tiles; ++it) {
                const int s = it % NB_STAGE;
                mbar_wait(bar_bempty(s), ((it / NB_STAGE) & 1u) ^ 1u);
                mbar_expect_tx(bar_bfull(s), TILE_BYTES);
                bulk_g2s(base + OFF_B + s * TILE_BYTES, b_tiles + (int64_t)it * TILE_BYTES, TILE_BYTES, bar_bfull(s));
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {  // MMA issue: 8 x (M128, N128, K16) per item tile
            mbar_wait(bar_a(), 0);
            for (int it = 0; it < n_item_tiles; ++it) {
                const int s = it % NB_STAGE, acc = it & 1;
                mbar_wait(bar_bfull(s), (it / NB_STAGE) & 1u);
                mbar_wait(bar_accempty(acc), ((it >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t d = tmem_base + (uint32_t)(acc * TN);
#pragma unroll
                for (int kh = 0; kh < 2; ++kh) {
                    const uint64_t da = umma_desc(base + OFF_A + kh * (TILE_BYTES / 2));
                    const uint64_t db = umma_desc(base + OFF_B + s * TILE_BYTES + kh * (TILE_BYTES / 2));
#pragma unroll
                    for (int k16 = 0; k16 < 4; ++k16)
                        umma_f16(d, da + (uint64_t)(k16 * 2), db + (uint64_t)(k16 * 2), IDESC_F16_M128_N128,
                                 (kh | k16) ? 1u : 0u);
                }
                tc_commit(bar_bempty(s));
                tc_commit(bar_accfull(acc));
            }
        }
    } else {
        // epilogue: thread = TMEM lane = user row; the scores never leave the SM
        const int64_t u = u0 + warp * 32 + lane;
        const bool live = u < ub;
        const int n_sub = n_item_tiles * (TN / SUB);
        float my_thr = 0.0f;
        int my_cnt = 0;  // this thread is the only writer of its user's candidate list: no atomics
        if (MODE == 1 && live) my_thr = thr[u];
        // cursor into the user's excluded ids: ex_next = ex_indices[ex], ex_after the one behind it (INT_MAX: none),
        // loaded one step ahead so that the walk rarely waits for a load
        int64_t ex = 0, ex_end = 0;
        int ex_next = INT_MAX, ex_after = INT_MAX;
        if (EXCL && live) {
            const int64_t user = users[u_begin + u];
            ex = ex_indptr[user];
            ex_end = ex_indptr[user + 1];
            if (ex < ex_end) ex_next = ex_indices[ex];
            if (ex + 1 < ex_end) ex_after = ex_indices[ex + 1];
        }
        for (int it = 0; it < n_item_tiles; ++it) {
            const int acc = it & 1;
            mbar_wait(bar_accfull(acc), (it >> 1) & 1u);
            tc_fence_after();
            const uint32_t t_row = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(acc * TN);
#pragma unroll 1
            for (int c = 0; c < TN / SUB; ++c) {
                uint32_t r[32];
                tmem_ld32(t_row + c * SUB, r);
                const int64_t col0 = (int64_t)it * TN + c * SUB;
                uint32_t xmask = 0;  // excluded columns of this block (duplicate ids set the same bit again)
                if (EXCL) {
                    const int c0 = (int)col0;  // ids are int32
                    while (ex_next < c0 + SUB) {
                        xmask |= 1u << (uint32_t)(ex_next - c0);
                        ex_next = ex_after;
                        ++ex;
                        ex_after = ex + 1 < ex_end ? ex_indices[ex + 1] : INT_MAX;
                    }
                }
                if (MODE == 0) {
                    float m = -3.0e38f;
                    if (EXCL) {  // branch-free: nearly every block has an excluded column in some lane of the warp
                        uint32_t keep = ~xmask;
                        if (col0 + SUB > ni) keep &= (col0 < ni) ? (0xFFFFFFFFu >> (32 - (int)(ni - col0))) : 0u;
#pragma unroll
                        for (int j = 0; j < SUB; ++j) m = fmaxf(m, ((keep >> j) & 1u) ? __uint_as_float(r[j]) : -3.0e38f);
                    } else if (col0 + SUB <= ni) {
#pragma unroll
                        for (int j = 0; j < SUB; ++j) m = fmaxf(m, __uint_as_float(r[j]));
                    } else {
#pragma unroll
                        for (int j = 0; j < SUB; ++j)
                            if (col0 + j < ni) m = fmaxf(m, __uint_as_float(r[j]));  // padding items never count
                    }
                    if (live) maxima[u * n_sub + it * (TN / SUB) + c] = m;
                } else if (live) {
                    uint32_t hits = 0;  // branch-free compare, then only the (rare) hits take the store path
#pragma unroll
                    for (int j = 0; j < SUB; ++j) hits |= (__uint_as_float(r[j]) >= my_thr ? 1u : 0u) << j;
                    if (col0 + SUB > ni) hits &= (col0 < ni) ? (0xFFFFFFFFu >> (32 - (int)(ni - col0))) : 0u;  // padding items
                    if (EXCL) hits &= ~xmask;
                    while (hits) {
                        const int j = __ffs(hits) - 1;
                        hits &= hits - 1;
                        if (my_cnt < CAND_MAX) lists[u * CAND_MAX + my_cnt] = (uint32_t)(col0 + j);
                        ++my_cnt;
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(bar_accempty(acc));
        }
        if (MODE == 1 && live) cnt[u] = my_cnt;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
    }
}

// thr[u] = (N-th largest block maximum) - 2 eps_u, one CTA per user (radix select in shared memory)
__global__ __launch_bounds__(128) void stc_threshold_kernel(const float* __restrict__ maxima, int n_sub, int topn,
                                                           const float* __restrict__ unorm,
                                                           const uint32_t* __restrict__ vmaxnorm, float* __restrict__ thr,
                                                           int* __restrict__ cnt) {
    extern __shared__ uint32_t skeys[];
    __shared__ unsigned hist[256];
    __shared__ unsigned s_prefix, s_need;
    const int tid = threadIdx.x;
    const float* row = maxima + (size_t)blockIdx.x * n_sub;
    for (int i = tid; i < n_sub; i += 128) skeys[i] = order_key(row[i]);
    unsigned prefix = 0, mask = 0, need = (unsigned)topn;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += 128) hist[i] = 0;
        __syncthreads();
        for (int i = tid; i < n_sub; i += 128) {
            const uint32_t k = skeys[i];
            if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid == 0) {
            unsigned acc = 0;
            int b = 255;
            for (; b > 0; --b) {
                if (acc + hist[b] >= need) break;
                acc += hist[b];
            }
            s_prefix = prefix | ((unsigned)b << shift);
            s_need = need - acc;
        }
        __syncthreads();
        prefix = s_prefix;
        need = s_need;
        mask |= 255u << shift;
        __syncthreads();
    }
    if (tid == 0) {
        const uint32_t tb = (prefix & 0x80000000u) ? (prefix & 0x7FFFFFFFu) : ~prefix;  // invert order_key
        const float tau = __uint_as_float(tb);
        const float eps = (1.02f * 0.0009765625f * unorm[blockIdx.x] * __uint_as_float(*vmaxnorm) + 0.25f) * 1.001f;
        thr[blockIdx.x] = tau - 2.0f * eps;
        cnt[blockIdx.x] = 0;
    }
}

// ---------------------------------------------------------------------------------------------------
// K5: exact rescoring of the candidates and the final top-N, one CTA per user
// ---------------------------------------------------------------------------------------------------
constexpr int TK_THREADS = 256;

// EXCL: a list shorter than topn is complete when the threshold is the -3e38 sentinel (fewer than topn unseen
// items: pass 2 admitted all of them); the rest of the row is id -1, score NaN. `fixup_users` (nullable) counts
// the users that make the exact path redo the call.
template <bool EXCL>
__global__ __launch_bounds__(TK_THREADS) void stc_rescore_kernel(
    const int* __restrict__ cnt, const uint32_t* __restrict__ lists, int topn, const int64_t* __restrict__ users,
    int64_t u_begin, const int64_t* __restrict__ cand, const float* __restrict__ U, int64_t ldu,
    const float* __restrict__ V, int64_t ldv, int f, int bias, int64_t* __restrict__ out_ids,
    float* __restrict__ out_scores, int* __restrict__ overflow, const float* __restrict__ thr,
    int* __restrict__ fixup_users) {
    __shared__ unsigned long long keys[CAND_MAX];
    __shared__ float su[K + 1];
    const int tid = threadIdx.x, lane = tid & 31;
    const int n_cand = cnt[blockIdx.x];
    const bool short_ok = EXCL && thr[blockIdx.x] <= -3.0e38f;
    if (n_cand > CAND_MAX || (n_cand < topn && !short_ok)) {  // too many near-ties for the candidate buffer: the exact path redoes the call
        if (tid == 0) {
            atomicOr(overflow, 1);
            if (EXCL && fixup_users) atomicAdd(fixup_users, 1);
        }
        return;
    }
    const uint32_t* cpos = lists + (size_t)blockIdx.x * CAND_MAX;
    // exact NumPy-order scores of the candidates (8 lanes per dot product)
    const float* ug = U + users[u_begin + blockIdx.x] * ldu;
    for (int i = tid; i < f; i += TK_THREADS) su[i] = ug[i];
    __syncthreads();
    const float* u = su;
    const int gl = lane & 7;
    const unsigned gmask = 0xFFu << (lane & 24);
    for (int c0 = 0; c0 < n_cand; c0 += TK_THREADS / 8) {
        const int c = c0 + (tid >> 3);
        const bool ok = c < n_cand;
        const uint32_t pos = cpos[ok ? c : 0];
        const float* v = V + (cand ? cand[pos] : (int64_t)pos) * ldv;
        float sc;
        if (f == 128 && !bias) {
            // np_block_sum for n = 128 with the 16 loads of this lane in flight together: accumulator gl takes
            // p[8b + gl], b = 0..15 in order, then ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) (wmf_model.py:206)
            float vv[16];
#pragma unroll
            for (int b = 0; b < 16; ++b) vv[b] = __ldg(v + 8 * b + gl);
            float r = __fmul_rn(u[gl], vv[0]);
#pragma unroll
            for (int b = 1; b < 16; ++b) r = __fadd_rn(r, __fmul_rn(u[8 * b + gl], vv[b]));
            r = __fadd_rn(r, __shfl_xor_sync(gmask, r, 1));
            r = __fadd_rn(r, __shfl_xor_sync(gmask, r, 2));
            r = __fadd_rn(r, __shfl_xor_sync(gmask, r, 4));
            sc = r;
        } else {
            sc = np_score(u, v, f, bias, gl, gmask);
        }
        if (ok && gl == 0) keys[c] = ((unsigned long long)order_key(sc) << 32) | (unsigned long long)(0xFFFFFFFFu - pos);
    }
    int npow = 1;
    while (npow < n_cand) npow <<= 1;
    for (int i = n_cand + tid; i < npow; i += TK_THREADS) keys[i] = 0ull;
    __syncthreads();
    for (int size = 2; size <= npow; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < npow / 2; t += TK_THREADS) {
                const int lo = 2 * t - (t & (stride - 1));
                const int hi = lo + stride;
                const bool desc = ((lo & size) == 0);
                const unsigned long long a = keys[lo], b = keys[hi];
                if ((a < b) == desc) { keys[lo] = b; keys[hi] = a; }
            }
            __syncthreads();
        }
    }
    for (int t = tid; t < topn; t += TK_THREADS) {
        if (EXCL && t >= n_cand) {
            out_ids[(size_t)blockIdx.x * topn + t] = -1;
            if (out_scores) out_scores[(size_t)blockIdx.x * topn + t] = __uint_as_float(0x7FFFFFFFu);
            continue;
        }
        const unsigned long long k = keys[t];
        const uint32_t pos = 0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFull);
        out_ids[(size_t)blockIdx.x * topn + t] = cand ? cand[pos] : (int64_t)pos;
        if (out_scores) {
            const uint32_t kb = (uint32_t)(k >> 32);
            out_scores[(size_t)blockIdx.x * topn + t] = __uint_as_float((kb & 0x80000000u) ? (kb & 0x7FFFFFFFu) : ~kb);
        }
    }
}

}  // namespace stc

using namespace stc;

bool score_tc_supported(int64_t ni, int f, int bias, int topn) {
    const int64_t n_sub = (ni + 127) / 128 * (TN / SUB);
    return (f + (bias ? 1 : 0)) <= K && ni >= 256 && topn <= 512 && topn <= ni / SUB && n_sub <= MAXSUB;
}

static inline int64_t pad128(int64_t x) { return (x + 127) / 128 * 128; }

int64_t score_tc_user_batch(int64_t nu) {  // two waves of 128-user CTAs per launch
    const int64_t cap = (int64_t)sm_count() * 2 * TM;
    return nu < cap ? nu : cap;
}

// layout of the tensor-core workspace (placed after the exact path's score tile)
struct TcLayout {
    size_t off_hdr, off_unorm, off_vnorm, off_thr, off_cnt, off_a, off_b, off_max, off_lists, total;
};
static TcLayout tc_layout(int64_t ubatch, int64_t ni) {
    TcLayout l;
    size_t o = 0;
    const size_t up = (size_t)pad128(ubatch), ip = (size_t)pad128(ni);
    l.off_hdr = o; o += 256;
    l.off_unorm = o; o += align_up(up * 4, 256);
    l.off_vnorm = o; o += align_up(ip * 4, 256);
    l.off_thr = o; o += align_up(up * 4, 256);
    l.off_cnt = o; o += align_up(up * 4, 256);
    l.off_a = o; o += up / 128 * TILE_BYTES;
    l.off_b = o; o += ip / 128 * TILE_BYTES;
    l.off_max = o; o += align_up(up * (ip / SUB) * 4, 256);
    l.off_lists = o; o += up * CAND_MAX * 4;
    l.total = o;
    return l;
}

size_t score_tc_workspace_bytes(int64_t nu, int64_t ni) { return tc_layout(score_tc_user_batch(nu), ni).total; }

// the block-maxima and candidate-list regions are dead once the tensor-core path has run: the exact fix-up
// (only executed after an overflow) uses them as its score tile
void score_tc_fixup_region(int64_t nu, int64_t ni, size_t* offset, size_t* bytes) {
    const TcLayout l = tc_layout(score_tc_user_batch(nu), ni);
    *offset = l.off_max;
    *bytes = l.total - l.off_max;
}

// One user batch of the tensor-core path; `ws` is the tensor-core part of the workspace. `overflow_flag`
// (device int) tells the caller's conditional exact kernels whether to redo the call.
int score_topk_tc_batch(const int64_t* users, int64_t u0, int ub, int64_t ubatch, const int64_t* cand, int64_t ni,
                        const float* U, int64_t ldu, const float* V, int64_t ldv, int f, int bias, int topn,
                        int64_t* out_ids, float* out_scores, void* ws, bool first_batch, int** overflow_flag,
                        cudaStream_t st, const int64_t* ex_indptr, const int32_t* ex_indices, int* fixup_users) {
    char* tc = reinterpret_cast<char*>(ws);
    const TcLayout l = tc_layout(ubatch, ni);
    uint32_t* hdr = reinterpret_cast<uint32_t*>(tc + l.off_hdr);  // [0] overflow, [1] absmax U, [2] absmax V, [3] max ||v~||
    float* unorm = reinterpret_cast<float*>(tc + l.off_unorm);
    float* vnorm = reinterpret_cast<float*>(tc + l.off_vnorm);
    float* thr = reinterpret_cast<float*>(tc + l.off_thr);
    int* cnt = reinterpret_cast<int*>(tc + l.off_cnt);
    uint8_t* a_tiles = reinterpret_cast<uint8_t*>(tc + l.off_a);
    uint8_t* b_tiles = reinterpret_cast<uint8_t*>(tc + l.off_b);
    float* maxima = reinterpret_cast<float*>(tc + l.off_max);
    uint32_t* lists = reinterpret_cast<uint32_t*>(tc + l.off_lists);
    *overflow_flag = reinterpret_cast<int*>(hdr);
    static bool attr_set = false;
    if (!attr_set) {
        WMF_CUDA(cudaFuncSetAttribute(stc_gemm_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        WMF_CUDA(cudaFuncSetAttribute(stc_gemm_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        WMF_CUDA(cudaFuncSetAttribute(stc_gemm_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        WMF_CUDA(cudaFuncSetAttribute(stc_gemm_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        attr_set = true;
    }
    const int sms = sm_count();
    const int n_tiles = (int)(pad128(ni) / 128), n_sub = n_tiles * (TN / SUB);
    if (first_batch) {  // item side and the overflow flag: once per call
        WMF_CUDA(cudaMemsetAsync(hdr, 0, 256, st));
        stc_absmax_kernel<<<sms * 2, 256, 0, st>>>(cand, 0, ni, V, ldv, f, hdr + 2);
        WMF_LAUNCH_CHECK("stc_absmax_kernel(items)");
        stc_convert_kernel<<<(unsigned)((pad128(ni) * 32 + 255) / 256), 256, 0, st>>>(cand, 0, ni, pad128(ni), V, ldv, f,
                                                                                       bias, 1, hdr + 2, b_tiles, vnorm);
        WMF_LAUNCH_CHECK("stc_convert_kernel(items)");
        stc_maxnorm_kernel<<<sms, 256, 0, st>>>(vnorm, ni, hdr + 3);
        WMF_LAUNCH_CHECK("stc_maxnorm_kernel");
    }
    WMF_CUDA(cudaMemsetAsync(hdr + 1, 0, 4, st));  // this batch's user maximum
    stc_absmax_kernel<<<sms * 2, 256, 0, st>>>(users, u0, ub, U, ldu, f, hdr + 1);
    WMF_LAUNCH_CHECK("stc_absmax_kernel(users)");
    const int64_t ub_pad = pad128(ub);
    stc_convert_kernel<<<(unsigned)((ub_pad * 32 + 255) / 256), 256, 0, st>>>(users, u0, ub, ub_pad, U, ldu, f, bias, 0,
                                                                               hdr + 1, a_tiles, unorm);
    WMF_LAUNCH_CHECK("stc_convert_kernel(users)");
    const unsigned grid = (unsigned)(ub_pad / 128);
    const bool excl = ex_indptr != nullptr;
    auto gemm0 = excl ? stc_gemm_kernel<0, true> : stc_gemm_kernel<0, false>;
    auto gemm1 = excl ? stc_gemm_kernel<1, true> : stc_gemm_kernel<1, false>;
    gemm0<<<grid, GEMM_THREADS, SMEM_BYTES, st>>>(a_tiles, b_tiles, n_tiles, ub, ni, maxima, nullptr, nullptr, nullptr,
                                                  users, u0, ex_indptr, ex_indices);
    WMF_LAUNCH_CHECK("stc_gemm_kernel<maxima>");
    stc_threshold_kernel<<<ub, 128, (size_t)n_sub * 4, st>>>(maxima, n_sub, topn, unorm, hdr + 3, thr, cnt);
    WMF_LAUNCH_CHECK("stc_threshold_kernel");
    gemm1<<<grid, GEMM_THREADS, SMEM_BYTES, st>>>(a_tiles, b_tiles, n_tiles, ub, ni, nullptr, thr, cnt, lists, users, u0,
                                                  ex_indptr, ex_indices);
    WMF_LAUNCH_CHECK("stc_gemm_kernel<filter>");
    auto rescore = excl ? stc_rescore_kernel<true> : stc_rescore_kernel<false>;
    rescore<<<ub, TK_THREADS, 0, st>>>(cnt, lists, topn, users, u0, cand, U, ldu, V, ldv, f, bias,
                                       out_ids + (size_t)u0 * topn, out_scores ? out_scores + (size_t)u0 * topn : nullptr,
                                       reinterpret_cast<int*>(hdr), thr, fixup_users);
    WMF_LAUNCH_CHECK("stc_rescore_kernel");
    return WMF_OK;
}

}  // namespace wmf
