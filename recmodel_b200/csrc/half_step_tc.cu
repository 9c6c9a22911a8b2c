// K2 (tcgen05 version): one ALS half-step for dim = 128, weighted, no bias.
// Replaces the per-row loop of recompute_factors (wmf_model.py:220-239).
//
// Per CSR row r:  A_r = G + sum_j d_j y_j y_j^T  (128x128, K = n_r),  b_r = sum_j (d_j+1) y_j,
// x_r = A_r^-1 b_r.  Everything O(f^2) per entry and O(f^3) per row runs on the 5th-gen tensor
// cores with FP32-equivalent accuracy (single-pass TF32/BF16 fails the 1e-4 bar, SURVEY.md D5):
//
//   Gram    z_j = S sqrt(d_j) y_j = zh + zl, both halves FP16 (11-bit significands, like TF32, but
//           K = 16 per instruction instead of 8); S is a power of two chosen per ROW from max diag(G)
//           (>= max y^2) and the row's max|d| so that zh never overflows FP16 and zl stays a normal
//           number for every entry that matters. W = sum zh zh^T + zh zl^T + zl zh^T: three
//           tcgen05.mma (kind::f16, M = N = 128, K = 16) per 16 stored entries into a 128-column
//           fp32 TMEM accumulator; operand tiles K-major, 128-byte swizzled.
//   Solve   block Gauss-Jordan, the matrix STAYS in TMEM. Steps of 8 columns: every thread
//           (= TMEM lane = matrix row) loads its 8 entries of the pivot columns (tcgen05.ld), adds G
//           lazily; the warp that owns the 8 pivot rows factors the 8x8 pivot block (straight-line
//           Cholesky in every lane, lane c then forms column c of L^-1) and publishes N = L^-1; every other row forms P = a N^T, updates its right-hand
//           side, writes P (TF32 hi/lo split) to shared memory as an MMA operand and the rank-8 update
//           S -= P P^T of ALL rows (above and below the pivots) is three tcgen05.mma (kind::tf32, negated
//           A, N trimmed to the live columns). After 16 steps the system is block diagonal and
//           x_blk = N^T N b_blk: no back substitution, nothing is written back to TMEM.
//
// TMEM holds four such matrices (4 x 128 = 512 columns): four solver groups of 128 threads each
// own one accumulator, so while one row is in its pivot chain three others fill the issue slots.
// One persistent CTA per SM, warp-specialised, all hand-offs through mbarriers:
//   warps 0-15  solve    group g = warp/4 owns accumulator g and the rows n with n % 4 == g.
//   warps 25-26 gather   one TMA producer warp per team: the 32 gathered factor rows of a sub-chunk land in a raw
//               staging buffer by eight cp.async.bulk.tensor ... tile::gather4 (TMA row gather, four 512-B rows per
//               instruction, completion on the buffer's mbarrier), two or three sub-chunks in flight per team
//   warps 16-23 transform two teams of 128 threads; a team takes every other 32-entry sub-chunk of a row. Thread m
//               owns feature m: it reads column m of the raw rows, scales, splits to FP16 hi/lo and stores the
//               K-major swizzled operand tiles a tiled TMA load would have produced (TMA cannot: the operand is
//               gathered, scaled and split); the rhs partial b[m] stays in registers.
//   warp 24     MMA      one thread issues the Gram MMAs (at most two K-steps queued, so the solvers'
//               rank-8 updates never wait behind a long burst) and commits stage/accumulator barriers.
//
// The tensor core truncates its fp32 accumulation, so a row with more than SPLIT_LEN entries is cut into
// segments that different CTAs accumulate; the group that parks the last segment adds the partial Grams in
// segment order (round-to-nearest) and solves the row (see the constants below and DESIGN.md 4.1).
//
// Rows whose weights are negative (sqrt undefined) or whose pivot block is not positive definite
// raise a flag; the caller then re-runs the half-step with the SIMT kernel (LU).
#include <stdlib.h>
#include <cuda.h>
#include <cudaTypedefs.h>
#include "tc_common.cuh"
#include "half_step.cuh"
#include "whiten.cuh"
#include "factor8.cuh"
#include "cg_solve.cuh"

namespace wmf {

namespace tc {

// operand stages / raw staging buffers per team: 4 / 3 or 6 / 2 fit the 227 KB (a row holds its accumulator for its
// Gram and its solve, so tiles staged ahead of a free accumulator shorten the Gram phase; the TMA row gathers want
// their own depth: a gather is in flight for ~1400 cycles when it misses L2, scripts/probe/tma_gather4_probe.cu)
#ifndef WMF_TC_STAGES
#define WMF_TC_STAGES 4
#endif
constexpr int STAGES = WMF_TC_STAGES, STAGING = STAGES == 4 ? 3 : 2;
static_assert(STAGES == 4 || STAGES == 6, "operand stages");

constexpr int F = 128;               // factor width handled by this kernel
constexpr int SUB = 32;              // stored entries per sub-chunk (one pipeline stage)
constexpr int NSTAGE = STAGES;       // operand stages (two sub-chunks share one 128-byte-swizzled tile pair)
constexpr int NTEAM = 2;             // gather teams (a TMA producer warp + four transform warps each)
constexpr int NSTG = STAGING;        // raw staging buffers per team (TMA gathers in flight)
constexpr int TILE_BYTES = F * 128;  // 128 rows (features) x 64 fp16 (K) = 16 KB, holds two sub-chunks
constexpr int PAIR_BYTES = 2 * TILE_BYTES;   // [zh ; zl]
constexpr int STG_BYTES = SUB * F * 4;       // 32 gathered factor rows, row-major fp32, 16 KB
constexpr int META_BYTES = SUB * 8 + 16;     // per staging buffer: S*sqrt(d) [32], (unused) [32], then the sub-chunk's descriptor
constexpr int NB = 8;                // Gauss-Jordan step width
// A operands of the Gram MMAs from tensor memory (WMF_TC_A_TMEM, default): the transform thread of feature m holds
// exactly row m of the K-major A tiles in registers, so it stores them into TMEM lane m (tcgen05.st) and only the
// B operands are read from shared memory: 12 KB instead of 24 KB per 16 entries on the resource that bounds this
// kernel. The four operand stages take 128 TMEM columns, which leaves three accumulators (systems in flight).
#ifndef WMF_TC_A_TMEM
#define WMF_TC_A_TMEM 1
#endif
constexpr bool A_TMEM = WMF_TC_A_TMEM != 0;
constexpr int NGROUP = A_TMEM ? 3 : 4;   // solver groups = TMEM accumulators
constexpr int OPND_COL0 = NGROUP * 128;  // first TMEM column of the A-operand stages (32 columns each: hi 16 | lo 16)
constexpr int GROUP = 128;
constexpr int TEAM = 128;
#ifndef WMF_TC_SOLVERS_FIRST
#define WMF_TC_SOLVERS_FIRST 1
#endif
// warp ids of the roles (solver warps start at a multiple of 4: warp id mod 4 is the TMEM lane quarter)
constexpr int GATHER_WARP0 = WMF_TC_SOLVERS_FIRST ? NGROUP * 4 : 0, SOLVER_WARP0 = WMF_TC_SOLVERS_FIRST ? 0 : NTEAM * 4;
constexpr int MMA_WARP = (NGROUP + NTEAM) * 4;
constexpr int PRODUCER_WARP0 = MMA_WARP + 1;               // one TMA producer warp per gather team
constexpr int THREADS = (PRODUCER_WARP0 + NTEAM) * 32;     // 864
constexpr uint32_t TMEM_COLS = 512;
constexpr int CG_BAR0 = 1 + NGROUP;  // named barriers 1 .. NGROUP: a whole solver group; CG_BAR0 + g: its warps that hold rows
static_assert(NGROUP * F + (A_TMEM ? NSTAGE * 32 : 0) <= 512, "TMEM columns");

// per-group shared memory
constexpr int PANEL_TILE_BYTES = F * NB * 4;          // 4 KB: 128 rows x 8 fp32, K-major, no swizzle
constexpr int G_OFF_TILEH = 0;
constexpr int G_OFF_TILEL = G_OFF_TILEH + PANEL_TILE_BYTES;
constexpr int G_OFF_NINV = G_OFF_TILEL + PANEL_TILE_BYTES;          // 16 blocks x (8 x 8) floats: N = L^-1 per pivot block
constexpr int G_OFF_ZB = G_OFF_NINV + (F / NB) * NB * NB * 4;       // 16 x 8 floats: N b_blk
constexpr int G_OFF_DBLK = G_OFF_ZB + (F / NB) * NB * 4;            // 8 x 8 pivot block + 8 rhs
constexpr int G_OFF_BFIN = G_OFF_DBLK + (NB * NB + 2 * NB) * 4;     // 128 floats: final rhs
constexpr int GROUP_BYTES = ((G_OFF_BFIN + F * 4 + 127) / 128) * 128;

// shared memory carve-up (bytes from a 1024-aligned base)
constexpr int OFF_STAGES = 0;                                        // NSTAGE/2 tile pairs
constexpr int OFF_STG = OFF_STAGES + (NSTAGE / 2) * PAIR_BYTES;
constexpr int OFF_META = OFF_STG + NTEAM * NSTG * STG_BYTES;
constexpr int OFF_GROUPS = ((OFF_META + NTEAM * NSTG * META_BYTES + 127) / 128) * 128;
constexpr int OFF_BVEC = OFF_GROUPS + NGROUP * GROUP_BYTES;         // NGROUP x NTEAM x F floats
constexpr int OFF_BARS = OFF_BVEC + NGROUP * NTEAM * F * 4;         // mbarriers (8 B each)
constexpr int NBARS = 2 * NSTAGE + 2 * NTEAM * NSTG + 2 + (4 + NTEAM) * NGROUP;
constexpr int OFF_TMEM_PTR = OFF_BARS + NBARS * 8;
constexpr int SMEM_BYTES = OFF_TMEM_PTR + 16 + 1024;                // + slack for alignment
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(OFF_GROUPS % 128 == 0 && GROUP_BYTES % 128 == 0 && OFF_BARS % 8 == 0 && OFF_STG % 1024 == 0, "alignment");

// workspace layout: see TcLayout below
constexpr size_t WS_PROF = 256, WS_TABLES = 1024;
// Rows longer than this are cut into segments of at most this many entries, for balance (a row never costs its
// CTA more than one segment) and for accuracy: the tensor core TRUNCATES its fp32 accumulation
// (scripts/probe/mma_round_probe.cu), a bias of ~half an ulp per MMA that grows with the number of MMAs into one
// accumulator. The segment partials are summed with round-to-nearest FP32 adds in segment order by the group that
// parks the last one. Environment knobs, read once per process (experiments; the defaults are the product):
//   WMF_TC_SPLIT=<entries>   segment length (default 2048)
//   WMF_TC_DUAL=0            send short rows to the primal kernel as well (dual kernel off)
//   WMF_TC_PROFILE=1         per-role cycle counters of CTA 0 (only in a -DWMF_TC_PROFILE_BUILD library)
constexpr int SPLIT_LEN_DEFAULT = 2048;
static int env_int_once(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }
static int split_len() {
    static const int v = [] { int x = env_int_once("WMF_TC_SPLIT", SPLIT_LEN_DEFAULT); if (x < 64) x = SPLIT_LEN_DEFAULT; return (x + 31) / 32 * 32; }();
    return v;
}
}  // namespace tc
// 64 products cover condition numbers up to ~100 (weights in the hundreds); beyond that the factorisation is cheaper
int tc_cg_max_products() {
    static const int v = [] { int x = tc::env_int_once("WMF_TC_CG", 64); return x < 0 ? 0 : (x > 1000 ? 1000 : x); }();
    return v;
}
namespace tc {
static bool dual_enabled() { static const bool v = env_int_once("WMF_TC_DUAL", 1) != 0; return v; }
static bool profile_enabled() {
#ifdef WMF_TC_PROFILE_BUILD
    static const bool v = env_int_once("WMF_TC_PROFILE", 0) != 0;
    return v;
#else
    return false;
#endif
}
constexpr int DEFAULT_PARTS = 2048;  // partial slots the legacy workspace query (rows only) provides
constexpr size_t PART_FLOATS = (size_t)F * F + F;  // a segment's S^2 W (chunk-major) and its rhs partial
constexpr int PACK_CHUNK = 1024;   // schedule slots per dual-row counter quad (tc_prep_rows_kernel, tc_pack_dual_kernel)
// ---------------------------------------------------------------------------------------------------
// prep: the schedule tables (one 16-byte entry per slot and kernel), the per-row FP16 scale, zero rows
// without entries, and the fix-up list.
// ---------------------------------------------------------------------------------------------------
// One warp per schedule slot. A row goes to exactly one place:
//   no stored entries              -> its whitened solution is zeroed here (wmf_model.py:223-225)
//   a negative weight (bias formula, d~ = d - beta, wmf_model.py:343), or G itself not positive definite
//                                  -> fix-up list: the CUDA-core LU kernel solves it after the tensor-core kernels
//   at most nd_max entries         -> dual table (half_step_dual.cu: n x n system)
//   otherwise                      -> primal table (f x f system: this file for f <= 128, half_step_tc256.cu above)
// Rows longer than SPLIT_LEN are cut into equal segments (a function of the row length only, so a row's
// arithmetic never depends on the launch it is in): segment 0 stays in the row's slot, the others go to
// extra slots behind the schedule, which the persistent CTAs reach round-robin like every other slot.
// Dual rows are also counted per chunk of PACK_CHUNK slots and per size class (32-lane TMEM slices: 1 ... 4) for the
// pack table (tc_pack_dual_kernel).
__global__ void tc_prep_rows_kernel(HalfStepParams p, int4* __restrict__ tab, int4* __restrict__ segtab,
                                    int4* __restrict__ dtab, uint32_t* __restrict__ pcnt, uint32_t* __restrict__ hdr_u,
                                    int64_t extra_slot0, int max_extra, int max_parts, int SPLIT_LEN, int primal_ok) {
    const int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __shared__ int64_t sh_lo[8], sh_hi[8];
    __shared__ float sh_m[8][8];
    __shared__ int sh_f[8][8];
    const int64_t row = s < p.sched_len ? (p.row_order ? (int64_t)p.row_order[s] : s) : -1;
    int64_t lo = 0, hi = 0;
    if (row >= 0) { lo = p.indptr[row]; hi = p.indptr[row + 1]; }
    // largest |weight| of the row, and whether a weight is negative (or NaN) / exactly zero. `stride` lanes walk the
    // row with eight loads in flight each.
    auto scan = [&](int64_t from, int64_t to, int first, int stride, float& m, int& flg) {
        for (int64_t i0 = from + first; i0 < to; i0 += (int64_t)stride * 8) {
            float d[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int64_t i = i0 + (int64_t)stride * u;
                d[u] = i < to ? __ldg(p.data + i) : 1.0f;
            }
            if (p.bias) {
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int64_t i = i0 + (int64_t)stride * u;
                    if (i < to) d[u] = __fsub_rn(d[u], __ldg(p.Yraw + (int64_t)__ldg(p.indices + i) * p.ldraw));
                }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (i0 + (int64_t)stride * u < to) {
                    flg |= (!(d[u] >= 0.0f) ? 1 : 0) | (d[u] == 0.0f ? 2 : 0);   // NaN weights go to the LU kernel too
                    m = fmaxf(m, fabsf(d[u]));
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            flg |= __shfl_xor_sync(0xffffffffu, flg, o);
        }
    };
    // Rows of up to COOP entries are scanned by their own warp; longer ones (they sit together at the head of a
    // longest-first schedule) by the whole block, one after the other: the longest row of the matrix is this kernel's
    // critical path (110 591 entries at ML-20M shape: 0.32 ms with one warp).
    constexpr int COOP = 1024;
    const bool big = hi - lo > COOP;
    float m = 0.0f;
    int flg = 0;
    if (!big) scan(lo, hi, lane, 32, m, flg);
    if (lane == 0) { sh_lo[w] = lo; sh_hi[w] = big ? hi : lo; }
    __syncthreads();
    for (int ww = 0; ww < 8; ++ww) {
        const int64_t l = sh_lo[ww], h = sh_hi[ww];
        if (h <= l) continue;  // uniform over the block
        float m2 = 0.0f;
        int f2 = 0;
        scan(l, h, threadIdx.x, 256, m2, f2);
        if (lane == 0) { sh_m[ww][w] = m2; sh_f[ww][w] = f2; }
    }
    __syncthreads();
    if (big) {
#pragma unroll
        for (int k = 0; k < 8; ++k) { m = fmaxf(m, sh_m[w][k]); flg |= sh_f[w][k]; }
    }
    if (s >= p.sched_len) return;
    int4 e = make_int4(-1, 0, 0, 0), de = make_int4(-1, 0, 0, 0);
    if (row >= 0) {
        int64_t n = hi - lo;
        const bool neg = (flg & 1) != 0, zero = (flg & 2) != 0;
        const bool g_bad = (hdr_u[1] & 8u) != 0;
        // the dual right-hand side (d+1)/sqrt(d) needs d > 0: a stored zero weight (it still adds y to the
        // right-hand side, wmf_model.py:239) keeps the row on the primal side
        const bool dual = n > 0 && n <= p.nd_max && !zero;
        if (n > 0 && (neg || g_bad || (!dual && !primal_ok))) {
            if (lane == 0) p.fix_list[atomicAdd(p.fix_count, 1)] = (int)row;
            n = -1;  // neither kernel touches it; the unwhitening pass writes zeros that the LU kernel overwrites
        }
        const int sexp = gram_scale_exp(__uint_as_float(hdr_u[2]), m);
        const uint32_t sbits = (uint32_t)(sexp + 64) << 16;
        e.x = de.x = (int32_t)row;
        if (n <= 0) {
            float4* x = reinterpret_cast<float4*>(p.X + row * p.ldx);  // whitened solution: ld = FP, 16-byte aligned
            for (int i = lane; i < p.FP / 4; i += 32) x[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        } else if (dual) {
            if (lane == 0) {
                atomicMax(hdr_u + 10, 0x7fffffffu - (uint32_t)s);
                atomicMax(hdr_u + 11, (uint32_t)s + 1u);
                atomicAdd(pcnt + (s / PACK_CHUNK) * 4 + (dual_slices((int)n) - 1), 1u);
            }
            de.y = (int32_t)n;
            de.z = (int32_t)(uint32_t)lo;
            de.w = (int32_t)((uint32_t)((lo >> 32) & 0xFFFF) | sbits);
        } else {
            if (lane == 0) atomicMax(hdr_u + 9, (uint32_t)s + 1u);
            // equal segments of whole sub-chunks, none empty (a function of the row length alone)
            int nseg = 1;
            int64_t seg_len = n;
            if (n > SPLIT_LEN) {
                const int64_t want = (n + SPLIT_LEN - 1) / SPLIT_LEN;
                seg_len = ((n + want - 1) / want + SUB - 1) / SUB * SUB;
                nseg = (int)((n + seg_len - 1) / seg_len);
            }
            int split_id = 0, first_part = 0, extra_base = 0;
            if (nseg > 1) {
                if (lane == 0) {
                    split_id = (int)atomicAdd(hdr_u + 5, 1u);
                    first_part = (int)atomicAdd(hdr_u + 6, (uint32_t)nseg);
                    extra_base = (int)atomicAdd(hdr_u + 7, (uint32_t)(nseg - 1));
                }
                split_id = __shfl_sync(0xffffffffu, split_id, 0);
                first_part = __shfl_sync(0xffffffffu, first_part, 0);
                extra_base = __shfl_sync(0xffffffffu, extra_base, 0);
                if (2 * split_id + 2 > max_parts || first_part + nseg > max_parts || extra_base + nseg - 1 > max_extra)
                    nseg = 1;  // out of scratch: the row stays whole (its CTA carries it alone; accuracy is unaffected
                               // at these lengths since the factors are whitened)
            }
            if (nseg == 1) {
                e.y = (int32_t)n;
                e.z = (int32_t)(uint32_t)lo;
                e.w = (int32_t)((uint32_t)((lo >> 32) & 0xFFFF) | sbits);
            } else {
                for (int k = lane; k < nseg; k += 32) {
                    const int64_t slo = lo + (int64_t)k * seg_len;
                    const int64_t shi = slo + seg_len < hi ? slo + seg_len : hi;
                    int4 se;
                    se.x = (int32_t)row;
                    se.y = (int32_t)(shi > slo ? shi - slo : 0);
                    se.z = (int32_t)(uint32_t)slo;
                    se.w = (int32_t)((uint32_t)((slo >> 32) & 0xFFFF) | sbits | 0x80000000u);  // bit 31: segment of a split row
                    const int64_t slot = k == 0 ? s : extra_slot0 + extra_base + (k - 1);
                    tab[slot] = se;
                    segtab[slot] = make_int4(split_id, nseg, first_part, k);
                }
                if (lane == 0) dtab[s] = de;
                return;
            }
        }
    }
    if (lane == 0) { tab[s] = e; dtab[s] = de; }
}

__device__ __forceinline__ uint4 add4u(uint4 a, uint4 b) { return make_uint4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ uint32_t get4u(uint4 a, int k) { return k == 0 ? a.x : k == 1 ? a.y : k == 2 ? a.z : a.w; }
__device__ __forceinline__ uint4 warp_scan4u(uint4 x) {   // inclusive
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint4 y = make_uint4(__shfl_up_sync(0xffffffffu, x.x, o), __shfl_up_sync(0xffffffffu, x.y, o),
                                   __shfl_up_sync(0xffffffffu, x.z, o), __shfl_up_sync(0xffffffffu, x.w, o));
        if (lane >= o) x = add4u(x, y);
    }
    return x;
}

// Packs of the dual kernel, longest first: every system of 4 slices alone; every 3-slice system with a 1-slice one
// from the short end of the 1-slice list while they last; the 2-slice systems in pairs, an odd one out with up to two
// more 1-slice systems; the remaining 1-slice systems in fours. With the dual rows of one size class in slot order
// (longest first on a sorted schedule), the row of rank i in class cls goes to (pack, first slice); `empty` gets
// the slices of that pack nobody takes when the row is its slice-0 system.
struct DualPackCounts {
    uint32_t c1, c2, c3, c4, m31, r1, p2, m21, r1b, packs;
    __device__ explicit DualPackCounts(const uint32_t* cnt) {
        c1 = cnt[0]; c2 = cnt[1]; c3 = cnt[2]; c4 = cnt[3];
        m31 = c1 < c3 ? c1 : c3;                   // 1-slice systems sharing a pack with a 3-slice one
        r1 = c1 - m31;
        p2 = (c2 + 1) / 2;
        m21 = (c2 & 1u) ? (r1 < 2u ? r1 : 2u) : 0u;   // 1-slice systems beside the odd 2-slice one
        r1b = r1 - m21;
        packs = c4 + c3 + p2 + (r1b + 3) / 4;
    }
    __device__ void place(int cls, uint32_t i, int64_t& pack, int& slice, uint32_t& empty) const {
        empty = 0;
        if (cls == 3) { pack = i; slice = 0; }
        else if (cls == 2) { pack = c4 + i; slice = 0; if (i >= m31) empty = 8u; }
        else if (cls == 1) {
            pack = c4 + c3 + i / 2; slice = 2 * (int)(i & 1u);
            if ((c2 & 1u) && i == c2 - 1) empty = (m21 < 1 ? 4u : 0u) | (m21 < 2 ? 8u : 0u);
        } else if (i >= r1) { pack = c4 + (c1 - 1 - i); slice = 3; }   // rank c1 - 1 - j joins 3-slice system j
        else if (i >= r1b) { pack = c4 + c3 + p2 - 1; slice = 2 + (int)(r1 - 1 - i); }
        else {
            pack = c4 + c3 + p2 + i / 4; slice = (int)(i & 3u);
            if (slice == 0)
                for (uint32_t k = 1; k < 4; ++k) if (i + k >= r1b) empty |= 1u << k;
        }
    }
};

// total slots = schedule (rounded up to a multiple of the grid) + extra segment slots. The per-chunk dual-row counts
// become exclusive prefixes per size class (in place); the class totals go to hdr[14 .. 17], the number of packs to hdr[13].
__global__ void __launch_bounds__(1024) tc_finish_prep_kernel(uint32_t* __restrict__ hdr_u, int64_t extra_slot0, int max_extra,
                                                              uint4* __restrict__ pcnt, int nchunks) {
    __shared__ uint4 wsum[32];
    __shared__ uint4 carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        const uint32_t extra = hdr_u[7] < (uint32_t)max_extra ? hdr_u[7] : (uint32_t)max_extra;
        hdr_u[4] = (uint32_t)(extra_slot0 + extra);
        carry = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    for (int c0 = 0; c0 < nchunks; c0 += 1024) {
        const int c = c0 + tid;
        const uint4 v = c < nchunks ? pcnt[c] : make_uint4(0u, 0u, 0u, 0u);
        const uint4 x = warp_scan4u(v);
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) wsum[lane] = warp_scan4u(wsum[lane]);
        __syncthreads();
        uint4 ex = add4u(carry, make_uint4(x.x - v.x, x.y - v.y, x.z - v.z, x.w - v.w));
        if (warp > 0) ex = add4u(ex, wsum[warp - 1]);
        if (c < nchunks) pcnt[c] = ex;
        __syncthreads();
        if (tid == 0) carry = add4u(carry, wsum[31]);
        __syncthreads();
    }
    if (tid == 0) {
        const uint32_t cnt[4] = {carry.x, carry.y, carry.z, carry.w};
        for (int k = 0; k < 4; ++k) hdr_u[14 + k] = cnt[k];
        hdr_u[13] = DualPackCounts(cnt).packs;
    }
}

// One block per chunk of the schedule: each dual row gets its rank in its size class (slot order: chunk prefix, then
// warps, then lanes) and from it its place in the pack table; its entry is written to every slice it covers.
__global__ void __launch_bounds__(PACK_CHUNK) tc_pack_dual_kernel(const int4* __restrict__ dtab, const uint4* __restrict__ pcnt,
                                                                  const uint32_t* __restrict__ hdr_u, int4* __restrict__ ptab,
                                                                  int64_t sched_len) {
    __shared__ uint32_t wcnt[PACK_CHUNK / 32][4];
    const int64_t s = (int64_t)blockIdx.x * PACK_CHUNK + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int4 de = s < sched_len ? dtab[s] : make_int4(-1, 0, 0, 0);
    const int cls = de.y > 0 ? dual_slices(de.y) - 1 : -1;
    uint32_t rank = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t m = __ballot_sync(0xffffffffu, cls == k);
        if (lane == 0) wcnt[warp][k] = __popc(m);
        if (cls == k) rank = __popc(m & ((1u << lane) - 1u));
    }
    __syncthreads();
    if (cls < 0) return;
    for (int w = 0; w < warp; ++w) rank += wcnt[w][cls];
    rank += get4u(pcnt[blockIdx.x], cls);
    const DualPackCounts pc(hdr_u + 14);
    int64_t pack;
    int slice;
    uint32_t empty;
    pc.place(cls, rank, pack, slice, empty);
    int4 ent = de;
    ent.w = (int32_t)((uint32_t)ent.w | ((uint32_t)slice << 24));
    for (int k = 0; k <= cls; ++k) ptab[pack * 4 + slice + k] = ent;
    for (int k = 1; k < 4; ++k)
        if (empty & (1u << k)) ptab[pack * 4 + k] = make_int4(-1, 0, 0, 0);
}

}  // namespace tc

using namespace tc;

template <bool PROF>
__global__ void __launch_bounds__(THREADS, 1)
als_half_step_tc_kernel(const __grid_constant__ CUtensorMap ymap, HalfStepParams p, const int4* __restrict__ rowtab,
                        const int4* __restrict__ segtab, float* __restrict__ parts, int* __restrict__ counters,
                        const uint32_t* __restrict__ hdr_u, int64_t extra_slot0, int* __restrict__ flags) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = smem_base + OFF_BARS;
    auto bar_full = [&](int s) { return bars + 8u * s; };
    auto bar_empty = [&](int s) { return bars + 8u * (NSTAGE + s); };
    auto bar_stg_full = [&](int team, int s) { return bars + 8u * (2 * NSTAGE + team * NSTG + s); };
    auto bar_stg_empty = [&](int team, int s) { return bars + 8u * (2 * NSTAGE + NTEAM * NSTG + team * NSTG + s); };
    auto bar_thr = [&](int x) { return bars + 8u * (2 * NSTAGE + 2 * NTEAM * NSTG + x); };
    constexpr int B0 = 2 * NSTAGE + 2 * NTEAM * NSTG + 2;
    auto bar_acc_full = [&](int g) { return bars + 8u * (B0 + g); };
    auto bar_acc_empty = [&](int g) { return bars + 8u * (B0 + NGROUP + g); };
    auto bar_b_empty = [&](int g) { return bars + 8u * (B0 + 2 * NGROUP + g); };
    auto bar_panel = [&](int g) { return bars + 8u * (B0 + 3 * NGROUP + g); };
    auto bar_b_full = [&](int g, int team) { return bars + 8u * (B0 + 4 * NGROUP + g * NTEAM + team); };

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(bar_full(s), TEAM); mbar_init(bar_empty(s), 1); }
        for (int s = 0; s < NTEAM * NSTG; ++s) { mbar_init(bar_stg_full(0, s), 1); mbar_init(bar_stg_empty(0, s), 4); }
        mbar_init(bar_thr(0), 1);
        mbar_init(bar_thr(1), 1);
        for (int g = 0; g < NGROUP; ++g) {
            mbar_init(bar_acc_full(g), 1);
            mbar_init(bar_acc_empty(g), GROUP);
            mbar_init(bar_b_empty(g), GROUP);
            mbar_init(bar_panel(g), 1);
            for (int tm = 0; tm < NTEAM; ++tm) mbar_init(bar_b_full(g, tm), TEAM);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const uint32_t tmem_ptr_addr = smem_base + OFF_TMEM_PTR;
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr),
                     "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_ptr_addr));

    // This CTA walks the slots s with s % gridDim == blockIdx: first the extra slots (segments of split rows,
    // behind the schedule in the table), then the schedule itself, so the long rows are merged early and
    // the tail of the kernel is made of short rows.
    const int ts = (int)gridDim.x;
    const int total_slots = (int)hdr_u[4];  // schedule + extra segment slots (set by the prep kernels), < 2^31
    const int nextra = (total_slots - (int)extra_slot0 - (int)blockIdx.x + ts - 1) / ts;
    // schedule slots at and beyond hdr[9] hold no row of this kernel (longest-first schedules put the short rows of
    // the dual kernel and the empty rows last): nobody walks them
    const int sched_end = min((int)extra_slot0, ((int)hdr_u[9] + ts - 1) / ts * ts);
    const int nslots = nextra + (sched_end - (int)blockIdx.x + ts - 1) / ts;
    const int base_x = (int)extra_slot0 + (int)blockIdx.x, base_s = (int)blockIdx.x - nextra * ts;
    auto ent_at = [&](int k) -> RowEnt {
        RowEnt e{-1, 0, 0, 0, -1};
        if (k < nslots) {
            const int slot = k * ts + (k < nextra ? base_x : base_s);
            e = unpack_ent(__ldg(rowtab + slot), slot);  // a segment's record sits at the same slot of the split table
        }
        return e;
    };

    if (warp >= PRODUCER_WARP0) {
        // =============================== GATHER: TMA PRODUCER ===============================
        // One warp per team. It walks the rows of this CTA, takes the sub-chunks c with (c + row_n) mod NTEAM == T and, for
        // each, has the 32 gathered factor rows copied into one of the team's raw staging buffers by the TMA unit:
        // eight cp.async.bulk.tensor ... tile::gather4 (four rows of 512 B each, lanes 0-7 issue one apiece) that
        // complete on the buffer's mbarrier. Beside the rows it leaves the per-entry scales S*sqrt(d), d+1 and a
        // descriptor (global sub-chunk index, row, last-of-row flag), so the eight transform warps run no cursor,
        // address or copy code at all. Entry indices and weights are loaded one step ahead; nothing may depend on
        // those loads in the step that issues them (a dependent instruction there parks the warp on the full
        // global-load latency every step).
        const int team = warp - PRODUCER_WARP0;
        int cu_k = -1;        // CTA-local slot of the current row
        int cu_row_n = -1;    // index of the row among this CTA's non-empty rows
        int cu_c = 0, cu_nsub = 0, cu_n = 0, cu_gi0 = 0;  // sub-chunk in row, sub-chunks / entries of the row, global index of sub-chunk 0
        int64_t cu_lo = 0;    // first entry of the row
        float cu_S = 1.0f;    // FP16 scale of the row
        RowEnt w0 = ent_at(0), w1 = ent_at(1);  // prefetched table entries k+1, k+2
        auto advance = [&](bool first) {  // to the team's next sub-chunk
            if (!first) cu_c += NTEAM;
            while (cu_k < nslots && cu_c >= cu_nsub) {
                bool found = false;
                while (!found) {  // next non-empty row
                    ++cu_k;
                    if (cu_k >= nslots) break;
                    const RowEnt e = w0;
                    w0 = w1;
                    w1 = ent_at(cu_k + 2);
                    if (e.n > 0) {
                        cu_gi0 += cu_nsub;
                        ++cu_row_n;
                        cu_n = e.n; cu_lo = e.lo; cu_nsub = (e.n + SUB - 1) / SUB; cu_S = exp2f((float)e.sexp);
                        found = true;
                    }
                }
                if (!found) break;
                cu_c = ((team - cu_row_n) % NTEAM + NTEAM) % NTEAM;   // the team takes the sub-chunks c with (c + row_n) % NTEAM == team
            }
        };
        struct Raw { int idx; float d; float s; int gi; int row_n; int last; };
        auto load_raw = [&]() {  // lane l: entry l of the cursor's sub-chunk
            Raw rw{-1, 0.f, cu_S, -1, 0, 0};
            if (cu_k < nslots) {
                rw.gi = cu_gi0 + cu_c; rw.row_n = cu_row_n; rw.last = cu_c + NTEAM >= cu_nsub ? 1 : 0;
                const int off = cu_c * SUB + lane;
                if (off < cu_n) {
                    rw.d = __ldg(p.data + cu_lo + off);      // loads only (see above)
                    rw.idx = __ldg(p.indices + cu_lo + off);
                }
            }
            return rw;
        };
        const int oob_row = (int)p.cols;   // a row index past the tensor: the TMA unit fills zeros (padding entries)
        advance(true);
        Raw nx = load_raw();
        uint32_t jp = 0;
        for (;;) {
            Raw rw = nx;
            if (rw.gi >= 0) { advance(false); nx = load_raw(); }
            const int buf = (int)(jp % NSTG);
            mbar_wait(bar_stg_empty(team, buf), ((jp / NSTG) & 1u) ^ 1u);   // the transform warps have read it
            const uint32_t mt = smem_base + OFF_META + (team * NSTG + buf) * META_BYTES;
            if (rw.gi < 0) {   // no more sub-chunks: leave the terminator
                if (lane == 0) { sts4u(mt + SUB * 8, 0xffffffffu, 0u, 0u, 0u); mbar_arrive(bar_stg_full(team, buf)); }
                break;
            }
            if (p.bias && rw.idx >= 0) rw.d = __fsub_rn(rw.d, __ldg(p.Yraw + (int64_t)rw.idx * p.ldraw));  // wmf_model.py:343
            {
                float sq = 0.f;
                if (rw.idx >= 0) sq = rw.s * sqrtf(rw.d);  // rows with a negative weight never get here (fix-up list, tc_prep_rows_kernel)
                sts1(mt + lane * 4, sq);
                if (lane == 0) sts4u(mt + SUB * 8, (uint32_t)rw.gi, (uint32_t)rw.row_n, (uint32_t)rw.last, __float_as_uint(1.0f / (rw.s * rw.s)));
            }
            const int vi = rw.idx >= 0 ? rw.idx : oob_row;
            const int i0 = __shfl_sync(0xffffffffu, vi, (4 * lane) & 31), i1 = __shfl_sync(0xffffffffu, vi, (4 * lane + 1) & 31);
            const int i2 = __shfl_sync(0xffffffffu, vi, (4 * lane + 2) & 31), i3 = __shfl_sync(0xffffffffu, vi, (4 * lane + 3) & 31);
            __syncwarp();   // every lane's scales are written before lane 0's release below
            const uint32_t fb = bar_stg_full(team, buf);
            if (lane == 0)
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fb), "r"((uint32_t)STG_BYTES) : "memory");
            if (lane < SUB / 4) {
                const uint32_t dst = smem_base + OFF_STG + (team * NSTG + buf) * STG_BYTES + lane * (4 * F * 4);
                asm volatile(
                    "cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes"
                    " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst), "l"(reinterpret_cast<uint64_t>(&ymap)), "r"(fb),
                    "r"(0), "r"(i0), "r"(i1), "r"(i2), "r"(i3) : "memory");
            }
            ++jp;
        }
    } else if (warp >= GATHER_WARP0 && warp < GATHER_WARP0 + NTEAM * 4) {
        // =============================== GATHER: TRANSFORM ===============================
        // Two teams of 128 threads; thread m owns feature m. A team takes the staging buffers its producer warp fills
        // in order: thread m reads column m of the 32 raw rows, scales, splits to FP16 hi/lo and stores the K-major
        // swizzled operand tiles a tiled TMA load would have produced (TMA cannot: the operand is gathered, scaled and
        // split); the rhs partial b[m] stays in registers until the row's last sub-chunk of the team.
        const int team = (warp - GATHER_WARP0) >> 2;
        const int m = (tid - GATHER_WARP0 * 32) & (TEAM - 1);  // feature index
        uint32_t j = 0;
        double bacc = 0.0;
        const bool prof = PROF && blockIdx.x == 0 && m == 0 && team == 0;
        long long t_empty = 0, t_bempty = 0, t_stg = 0, t_xform = 0, t_start = prof ? clock64() : 0, tt = 0, t2 = 0;
        for (;;) {
            const int sb = (int)(j % NSTG);
            if (prof) t2 = clock64();
            mbar_wait(bar_stg_full(team, sb), (j / NSTG) & 1u);   // rows (async proxy) and scales (producer warp) have landed
            if (prof) { tt = clock64(); t_stg += tt - t2; }
            const uint32_t stg = smem_base + OFF_STG + (team * NSTG + sb) * STG_BYTES + m * 4;
            const uint32_t mt = smem_base + OFF_META + (team * NSTG + sb) * META_BYTES;
            int d_gi, d_row_n, d_last;
            float d_inv_s2;
            {
                uint32_t a, b, c, d;
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(mt + SUB * 8));
                d_gi = (int)a; d_row_n = (int)b; d_last = (int)c; d_inv_s2 = __uint_as_float(d);
            }
            if (d_gi < 0) break;
            const int s = d_gi % NSTAGE;
            mbar_wait(bar_empty(s), (((uint32_t)d_gi / NSTAGE) & 1u) ^ 1u);
            if (prof) { t2 = clock64(); t_empty += t2 - tt; tt = t2; }
            if (A_TMEM) tc_fence_after();   // the MMAs that read this stage's TMEM operands have completed
            const uint32_t tile_h = smem_base + OFF_STAGES + (s >> 1) * PAIR_BYTES + m * 128;
            const uint32_t opnd = tmem_base + ((uint32_t)((m >> 5) * 32) << 16) + (uint32_t)(OPND_COL0 + s * 32);
            const int half = s & 1;
            // rhs partial: sum (d + 1) v = sum v + (1 / S^2) sum z sq  with z = sq v, sq = S sqrt(d) (one scale per entry
            // to read instead of two: this kernel is bound by shared-memory wavefronts)
            float part1 = 0.f, partd = 0.f;
            // The shared-memory accessors are volatile asm (program order is issue order), so the loads of chunk c+1
            // are written ahead of the arithmetic and stores of chunk c: one LDS latency is exposed per sub-chunk
            // instead of one per 8 entries.
            float vn[8], sqn[8];
            auto load_chunk = [&](int c) {
                const float4 sa = lds4(mt + c * 32), sb4 = lds4(mt + c * 32 + 16);
                sqn[0] = sa.x; sqn[1] = sa.y; sqn[2] = sa.z; sqn[3] = sa.w; sqn[4] = sb4.x; sqn[5] = sb4.y; sqn[6] = sb4.z; sqn[7] = sb4.w;
#pragma unroll
                for (int e = 0; e < 8; ++e) vn[e] = lds1(stg + (c * 8 + e) * (F * 4));
            };
            load_chunk(0);
#pragma unroll
            for (int c = 0; c < SUB / 8; ++c) {   // one 16-byte chunk = 8 entries of this feature
                float v[8], sq[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) { v[e] = vn[e]; sq[e] = sqn[e]; }
                if (c + 1 < SUB / 8) load_chunk(c + 1);
                uint32_t hh[4], ll[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float v0 = v[2 * e], v1 = v[2 * e + 1];
                    const float z0 = sq[2 * e] * v0, z1 = sq[2 * e + 1] * v1;
                    part1 += v0;
                    partd = fmaf(z0, sq[2 * e], partd);
                    part1 += v1;
                    partd = fmaf(z1, sq[2 * e + 1], partd);
                    const __half2 h = __floats2half2_rn(z0, z1);
                    const float2 hf = __half22float2(h);
                    const __half2 l = __floats2half2_rn(z0 - hf.x, z1 - hf.y);
                    hh[e] = h2_bits(h);
                    ll[e] = h2_bits(l);
                }
                const uint32_t sw = (uint32_t)(((half * 4 + c) ^ (m & 7)) << 4);  // 128B swizzle: chunk index XOR (row mod 8)
                sts4u(tile_h + sw, hh[0], hh[1], hh[2], hh[3]);
                sts4u(tile_h + TILE_BYTES + sw, ll[0], ll[1], ll[2], ll[3]);
                if (A_TMEM) {   // row m of the A tiles: K-step c / 2, words 4 (c & 1) .. of its 8 columns
                    tmem_st4(opnd + (uint32_t)(c * 4), hh[0], hh[1], hh[2], hh[3]);
                    tmem_st4(opnd + 16u + (uint32_t)(c * 4), ll[0], ll[1], ll[2], ll[3]);
                }
            }
            const float part = fmaf(partd, d_inv_s2, part1);
            if (A_TMEM) { tmem_wait_st(); tc_fence_before(); }
            bacc += (double)part;
            fence_async_smem();  // generic-proxy stores -> visible to the tensor core (async proxy)
            mbar_arrive(bar_full(s));
            __syncwarp();        // every lane has read the raw rows and scales: the producer may refill the buffer
            if (lane == 0) mbar_arrive(bar_stg_empty(team, sb));
            if (prof) { t2 = clock64(); t_xform += t2 - tt; }
            if (d_last) {  // hand the team's rhs partial to the solver group that owns this row
                const int g = d_row_n % NGROUP;
                const uint32_t bph = ((uint32_t)d_row_n / NGROUP) & 1u;
                mbar_wait(bar_b_empty(g), bph ^ 1u);
                sts1(smem_base + OFF_BVEC + ((g * NTEAM + team) * F + m) * 4, (float)bacc);
                mbar_arrive(bar_b_full(g, team));
                bacc = 0.0;
                if (prof) t_bempty += clock64() - t2;
            }
            ++j;
        }
        if (prof) { p.prof[0] = clock64() - t_start; p.prof[1] = t_empty; p.prof[2] = t_bempty; p.prof[3] = j; p.prof[5] = t_stg; p.prof[12] = t_xform; }
    } else if (warp == MMA_WARP) {
        // =============================== GRAM MMA ISSUE ===============================
        // The whole warp runs the (warp-uniform) loop and waits on the barriers; one elected lane issues the MMAs and
        // the commits (see elect_one()).
        {
            uint32_t gi = 0, row_n = 0;
            const bool prof = PROF && blockIdx.x == 0 && lane == 0;
            long long t_full = 0, t_accempty = 0, t_thr = 0, t_start = prof ? clock64() : 0, tt = 0;
            RowEnt nxt = ent_at(0);
            for (int k = 0; k < nslots; ++k) {
                const RowEnt e = nxt;
                nxt = ent_at(k + 1);
                if (e.n <= 0) continue;
                const int g = row_n % NGROUP;
                const uint32_t aph = (row_n / NGROUP) & 1u;
                if (prof) tt = clock64();
                mbar_wait(bar_acc_empty(g), aph ^ 1u);
                if (prof) t_accempty += clock64() - tt;
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(g * F);
                const uint32_t idesc_gram = IDESC_F16_M128 | ((uint32_t)(p.f16 >> 3) << 17);  // N = live columns
                uint32_t accumulate = 0;
                for (int base = 0; base < e.n; base += SUB, ++gi) {
                    const int s = gi % NSTAGE;
                    if (prof) tt = clock64();
                    mbar_wait(bar_full(s), (gi / NSTAGE) & 1u);
                    if (prof) t_full += clock64() - tt;
                    tc_fence_after();
                    const int kc = (e.n - base) < SUB ? (e.n - base) : SUB;
                    const uint32_t tile = smem_base + OFF_STAGES + (s >> 1) * PAIR_BYTES + (s & 1) * 64;
                    const uint64_t dh = umma_desc(tile), dl = umma_desc(tile + TILE_BYTES);
                    if (p.cg_maxit == 0 && gi >= 2) {  // factorisation only: at most two sub-chunks (12 MMAs) queued ahead of the solvers' rank-8 updates
                        if (prof) tt = clock64();
                        mbar_wait(bar_empty((gi - 2) % NSTAGE), ((gi - 2) / NSTAGE) & 1u);
                        if (prof) t_thr += clock64() - tt;
                    }
                    if (elect_one()) {
                        // 16 fp16 = 32 B along K inside the 128-B swizzle row per K-step; a sub-chunk is one or two of them
                        if (A_TMEM) {
                            const uint32_t ah = tmem_base + (uint32_t)(OPND_COL0 + s * 32), al = ah + 16u;
                            umma_f16_ts(d_tmem, ah, dh, idesc_gram, accumulate);  // zh zh^T
                            umma_f16_ts(d_tmem, ah, dl, idesc_gram, 1u);          // zh zl^T
                            umma_f16_ts(d_tmem, al, dh, idesc_gram, 1u);          // zl zh^T
                            if (kc > 16) {
                                umma_f16_ts(d_tmem, ah + 8u, dh + 2, idesc_gram, 1u);
                                umma_f16_ts(d_tmem, ah + 8u, dl + 2, idesc_gram, 1u);
                                umma_f16_ts(d_tmem, al + 8u, dh + 2, idesc_gram, 1u);
                            }
                        } else {
                            umma_f16(d_tmem, dh, dh, idesc_gram, accumulate);  // zh zh^T
                            umma_f16(d_tmem, dh, dl, idesc_gram, 1u);          // zh zl^T
                            umma_f16(d_tmem, dl, dh, idesc_gram, 1u);          // zl zh^T
                            if (kc > 16) {
                                umma_f16(d_tmem, dh + 2, dh + 2, idesc_gram, 1u);
                                umma_f16(d_tmem, dh + 2, dl + 2, idesc_gram, 1u);
                                umma_f16(d_tmem, dl + 2, dh + 2, idesc_gram, 1u);
                            }
                        }
                        tc_commit(bar_empty(s));
                    }
                    __syncwarp();
                    accumulate = 1;
                }
                if (elect_one()) tc_commit(bar_acc_full(g));
                __syncwarp();
                ++row_n;
            }
            if (prof) { p.prof[8] = clock64() - t_start; p.prof[9] = t_full; p.prof[10] = t_accempty; p.prof[13] = t_thr; }
        }
    } else {
        // =============================== SOLVE (matrix resident in TMEM) ===============================
        // Block Gauss-Jordan on the 128x128 system, 8 columns per step (see the header): no back
        // substitution and nothing is written back to TMEM.
        const int g = (warp - SOLVER_WARP0) >> 2;
        const int q = warp & 3;        // TMEM lane quarter this warp may access
        const int t = q * 32 + lane;   // matrix row owned by this thread = TMEM lane
        const int bar_id = 1 + g;
        const int ISSUE_T = 32 * g;  // thread of the group that issues its rank-8 update MMAs
        const uint32_t gs = smem_base + OFF_GROUPS + g * GROUP_BYTES;
        const uint32_t tileH = gs + G_OFF_TILEH, tileL = gs + G_OFF_TILEL;
        const uint32_t Nst = gs + G_OFF_NINV, zst = gs + G_OFF_ZB, Dblk = gs + G_OFF_DBLK, bfin = gs + G_OFF_BFIN;
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * F);
        const uint32_t d_tmem = tmem_base + (uint32_t)(g * F);
        const uint64_t descH = umma_desc_panel(tileH), descL = umma_desc_panel(tileL);
        const int f8 = p.f8, f16 = p.f16;  // live width: the whitened system is the identity beyond it
        // a warp whose 32 lanes lie beyond the live width (f <= 64: two of the four) owns no matrix row: it only keeps
        // the group's barriers (and, if it is warp g, the pivot factor) and skips the per-row work
        const bool active = q * 32 < f16;
        const int nact = (f16 + 31) >> 5;   // warps of the group that hold matrix rows
        uint32_t row_n = 0, panel_n = 0, b_phase = 0;
        const bool prof = PROF && blockIdx.x == 0 && g == 0 && t == 0;
        long long t_accfull = 0, t_fact = 0, t_back = 0, t_start = prof ? clock64() : 0, tt = 0;
        long long ph_wait = 0, ph_ld = 0, ph_own = 0, ph_p = 0, ph_issue = 0, t3 = 0, t4 = 0, my_rows = 0, cg_rows = 0, cg_products = 0;
        RowEnt nxt = ent_at(0);
        for (int k = 0; k < nslots; ++k) {
            const RowEnt e = nxt;
            nxt = ent_at(k + 1);
            if (e.n <= 0) continue;
            const uint32_t rn = row_n++;
            if ((int)(rn % NGROUP) != g) continue;
            ++my_rows;
            float* xout = p.X + (int64_t)e.row * p.ldx;
            const float S = exp2f((float)e.sexp), inv_s = exp2f((float)-e.sexp), inv_s2 = inv_s * inv_s;  // exact powers of two
            if (prof) tt = clock64();
            // rhs partials: one per residue class c mod NTEAM of the row's sub-chunks (class k is the work of team
            // (k + row_n) mod NTEAM), added in class order: a function of the row alone
            float bt = 0.0f;
            {
                const int nsub_row = (e.n + SUB - 1) / SUB;
#pragma unroll
                for (int cls = 0; cls < NTEAM; ++cls) {
                    if (cls < nsub_row) {
                        const int tm = (cls + (int)(rn % NTEAM)) % NTEAM;
                        mbar_wait(bar_b_full(g, tm), (b_phase >> tm) & 1u);
                        b_phase ^= 1u << tm;
                        const float bp = lds1(smem_base + OFF_BVEC + ((g * NTEAM + tm) * F + t) * 4);
                        bt = cls == 0 ? bp : bt + bp;
                    }
                }
            }
            mbar_arrive(bar_b_empty(g));
            mbar_wait(bar_acc_full(g), (rn / NGROUP) & 1u);
            tc_fence_after();
            if (prof) { t_accfull += clock64() - tt; tt = clock64(); }
            if (e.part >= 0) {
                // ---- segment of a split row: park the partial S^2 W and rhs in the scratch; the segment that arrives
                // last adds all of them in segment order (deterministic) and goes on to solve the row
                const int4 sg = __ldg(segtab + e.part);  // split_id, nseg, first_part, seg
                float* mine = parts + (size_t)(sg.z + sg.w) * PART_FLOATS;
#pragma unroll 1
                for (int c0 = 0; c0 < f8; c0 += NB) {
                    float a[NB];
                    tmem_ld8(t_row + c0, a);
                    float4* dst = reinterpret_cast<float4*>(mine + (c0 >> 3) * (F * NB) + t * NB);
                    dst[0] = make_float4(a[0], a[1], a[2], a[3]);
                    dst[1] = make_float4(a[4], a[5], a[6], a[7]);
                }
                mine[F * F + t] = bt;
                __threadfence();
                named_bar(bar_id, GROUP);
                if (t == 0) sts1(Dblk, __int_as_float(atomicAdd(counters + sg.x, 1) == sg.y - 1 ? 1 : 0));
                named_bar(bar_id, GROUP);
                const bool last = __float_as_int(lds1(Dblk)) != 0;
                named_bar(bar_id, GROUP);  // Dblk is reused by the solve below
                if (!last) {
                    tc_fence_before();
                    mbar_arrive(bar_acc_empty(g));
                    continue;
                }
                __threadfence();
                const float* first = parts + (size_t)sg.z * PART_FLOATS;
#pragma unroll 1
                for (int c0 = 0; c0 < f8; c0 += NB) {
                    float a[NB] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                    for (int k2 = 0; k2 < sg.y; ++k2) {
                        const float4* src = reinterpret_cast<const float4*>(first + (size_t)k2 * PART_FLOATS + (c0 >> 3) * (F * NB) + t * NB);
                        const float4 x0 = __ldcg(src), x1 = __ldcg(src + 1);
                        a[0] += x0.x; a[1] += x0.y; a[2] += x0.z; a[3] += x0.w;
                        a[4] += x1.x; a[5] += x1.y; a[6] += x1.z; a[7] += x1.w;
                    }
                    tmem_st8(t_row + c0, a);
                }
                bt = 0.0f;
                for (int k2 = 0; k2 < sg.y; ++k2) bt += __ldcg(first + (size_t)k2 * PART_FLOATS + F * F + t);
                tc_fence_before();
                named_bar(bar_id, GROUP);
                tc_fence_after();
            }
            // ---- default solver: conjugate gradients against the matrix in tensor memory (cg_solve.cuh). The block
            // Gauss-Jordan below takes the rows that have not converged within p.cg_maxit products (and every row when
            // p.cg_maxit == 0: WMF_ALGO_TCGEN05_DIRECT).
            if (p.cg_maxit > 0) {
                float xc = 0.0f;
                int products = -1;
                if (active) products = cg_solve(t_row, t, f16, bt, inv_s2, bfin, Dblk, q, nact, CG_BAR0 + g, nact * 32, p.cg_maxit, xc, prof ? p.prof + 48 : nullptr);
                const uint32_t flag = Dblk + 128u + (uint32_t)(my_rows & 1) * 4u;
                if (t == 0) sts1(flag, products >= 0 ? 1.0f : 0.0f);
                if (prof) { cg_rows += products >= 0; cg_products += products >= 0 ? products : p.cg_maxit + 1; }
                tc_fence_before();
                named_bar(bar_id, GROUP);
                if (lds1(flag) != 0.0f) {
                    mbar_arrive(bar_acc_empty(g));   // the Gram of this group's next row may start
                    xout[t] = t < f8 ? xc : 0.0f;
                    if (prof) t_fact += clock64() - tt;
                    continue;
                }
                                // header word 12: some row took the factorisation (a plain store: an atomicAdd at this point made the
                // whole kernel 50 % slower, measured A/B on one box, although it never executes on the bench workloads)
                if (t == 0) *reinterpret_cast<volatile int*>(flags + 11) = 1;

                tc_fence_after();
            }
#pragma unroll 1
            for (int c0 = 0; c0 < f8; c0 += NB) {
                if (prof) t3 = clock64();
                if (c0 > 0) {  // the previous step's rank-8 update has landed in TMEM
                    if (active) { mbar_wait(bar_panel(g), panel_n & 1u); tc_fence_after(); }
                    ++panel_n;
                }
                if (prof) { t4 = clock64(); ph_wait += t4 - t3; }
                float a[NB] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                if (active) tmem_ld8(t_row + c0, a);
                if (c0 + NB == f8) {  // last read of the accumulator: the Gram of this group's next row may start
                    tc_fence_before();
                    mbar_arrive(bar_acc_empty(g));
                }
                const int rel = t - c0;
#pragma unroll
                for (int i = 0; i < NB; ++i) a[i] = fmaf(a[i], inv_s2, rel == i ? 1.0f : 0.0f);  // I + sum d y~ y~^T
                if (prof) { t3 = clock64(); ph_ld += t3 - t4; }
                const uint32_t nd = Nst + (c0 >> 3) * 256, zd = zst + (c0 >> 3) * 32;
                // The 8 threads that hold the pivot rows publish them; the serial 8x8 factor is run by warp g of
                // group g, whatever warp the pivot rows live in: the four groups' serial chains then sit on four
                // different warp schedulers (warp id mod 4) instead of piling up on the scheduler of the quarter all
                // groups happen to be in (short dual rows never leave quarter 0).
                if (rel >= 0 && rel < NB) {
                    sts4(Dblk + rel * 32, a[0], a[1], a[2], a[3]);
                    sts4(Dblk + rel * 32 + 16, a[4], a[5], a[6], a[7]);
                    sts1(Dblk + 256 + rel * 4, bt);
                }
                named_bar(bar_id, GROUP);
                if (q == g) {
                    float d[36], bb[NB];
#pragma unroll
                    for (int i = 0; i < NB; ++i) {
                        const float4 d0 = lds4(Dblk + i * 32);
                        d[TRI(i, 0)] = d0.x;
                        if (i >= 1) d[TRI(i, 1)] = d0.y;
                        if (i >= 2) d[TRI(i, 2)] = d0.z;
                        if (i >= 3) d[TRI(i, 3)] = d0.w;
                        if (i >= 4) {
                            const float4 d1 = lds4(Dblk + i * 32 + 16);
                            d[TRI(i, 4)] = d1.x;
                            if (i >= 5) d[TRI(i, 5)] = d1.y;
                            if (i >= 6) d[TRI(i, 6)] = d1.z;
                            if (i >= 7) d[TRI(i, 7)] = d1.w;
                        }
                    }
                    {
                        const float4 b0 = lds4(Dblk + 256), b1 = lds4(Dblk + 272);
                        bb[0] = b0.x; bb[1] = b0.y; bb[2] = b0.z; bb[3] = b0.w;
                        bb[4] = b1.x; bb[5] = b1.y; bb[6] = b1.z; bb[7] = b1.w;
                    }
                    float ncol[NB], z[NB];
                    const bool ok = factor8(d, bb, lane & 7, ncol, z);  // lane c holds column c of N = L^-1
                    // published scaled: S N and z / S, so P comes out as S P (the MMA operand) for free
                    if (lane < NB) {
#pragma unroll
                        for (int i = 0; i < NB; ++i) sts1(nd + i * 32 + lane * 4, S * ncol[i]);
                    }
                    if (lane == 0) {
                        sts4(zd, inv_s * z[0], inv_s * z[1], inv_s * z[2], inv_s * z[3]);
                        sts4(zd + 16, inv_s * z[4], inv_s * z[5], inv_s * z[6], inv_s * z[7]);
                        if (!ok) {  // cannot happen with non-negative weights (spectrum >= 1); a numerical accident
                                    // sends the row to the LU kernel and leaves a host-visible mark
                            atomicOr(flags, 2);
                            p.fix_list[atomicAdd(p.fix_count, 1)] = e.row;
                        }
                    }
                    if (prof) { t4 = clock64(); ph_own += t4 - t3; }
                }
                named_bar(bar_id, GROUP);
                // ---- every row outside the block: P = a (S N)^T = S a N^T, rhs -= P (zb / S); the block's own rows
                // are pivots (P = 0) ----
                float P[NB] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                if (active) {
#pragma unroll
                    for (int jj = 0; jj < NB; ++jj) {
                        const float4 n0 = lds4(nd + jj * 32);
                        float v = a[0] * n0.x;
                        if (jj >= 1) v = fmaf(a[1], n0.y, v);
                        if (jj >= 2) v = fmaf(a[2], n0.z, v);
                        if (jj >= 3) v = fmaf(a[3], n0.w, v);
                        if (jj >= 4) {
                            const float4 n1 = lds4(nd + jj * 32 + 16);
                            v = fmaf(a[4], n1.x, v);
                            if (jj >= 5) v = fmaf(a[5], n1.y, v);
                            if (jj >= 6) v = fmaf(a[6], n1.z, v);
                            if (jj >= 7) v = fmaf(a[7], n1.w, v);
                        }
                        P[jj] = v;
                    }
                    if (q == (c0 >> 5)) {  // only the owner warp holds pivot rows
                        const bool pivot = rel >= 0 && rel < NB;
#pragma unroll
                        for (int jj = 0; jj < NB; ++jj) P[jj] = pivot ? 0.0f : P[jj];
                    }
                    const float4 z0 = lds4(zd), z1 = lds4(zd + 16);
                    float u0 = P[0] * z0.x, u1 = P[1] * z0.y;  // two chains, fixed order
                    u0 = fmaf(P[2], z0.z, u0); u1 = fmaf(P[3], z0.w, u1);
                    u0 = fmaf(P[4], z1.x, u0); u1 = fmaf(P[5], z1.y, u1);
                    u0 = fmaf(P[6], z1.z, u0); u1 = fmaf(P[7], z1.w, u1);
                    bt -= u0 + u1;
                }
                if (c0 + NB < f8) {
                    if (active) {
                        float lh[NB], ll[NB];
#pragma unroll
                        for (int jj = 0; jj < NB; ++jj) {  // the accumulator holds S^2 W: the update is (S P)(S P)^T
                            lh[jj] = tf32_round(P[jj]);
                            ll[jj] = P[jj] - lh[jj];  // exact; the tensor core reads its top 19 bits (error 2^-23 of P)
                        }
                        const uint32_t o = (uint32_t)((t >> 3) * 256 + (t & 7) * 16);
                        sts4(tileH + o, lh[0], lh[1], lh[2], lh[3]);
                        sts4(tileH + o + 128, lh[4], lh[5], lh[6], lh[7]);
                        sts4(tileL + o, ll[0], ll[1], ll[2], ll[3]);
                        sts4(tileL + o + 128, ll[4], ll[5], ll[6], ll[7]);
                        fence_async_smem();
                        tc_fence_before();
                    }
                    if (prof) t3 = clock64();
                    named_bar(bar_id, GROUP);
                    if (t == ISSUE_T) {
                        // S[:, j] -= P P[j]^T for the live columns j >= c0 + 8 (all 128 rows: Gauss-Jordan)
                        tc_fence_after();
                        if (prof) { t4 = clock64(); ph_p += t4 - t3; }
                        const uint32_t start = (uint32_t)((c0 + NB) >> 4) << 4;
                        const uint32_t idesc = IDESC_TF32_NEG_M128 | ((((uint32_t)f16 - start) >> 3) << 17);
                        const uint64_t bH = descH + (uint64_t)(start * 2), bL = descL + (uint64_t)(start * 2);
                        umma_tf32(d_tmem + start, descH, bH, idesc, 1u);
                        umma_tf32(d_tmem + start, descH, bL, idesc, 1u);
                        umma_tf32(d_tmem + start, descL, bH, idesc, 1u);
                        tc_commit(bar_panel(g));
                        if (prof) ph_issue += clock64() - t4;
                    }
                }
            }
            if (prof) { t_fact += clock64() - tt; tt = clock64(); }
            // ---- the system is block diagonal now: x_blk = (L L^T)^-1 b_blk = N^T (N b_blk) ----
            sts1(bfin + t * 4, bt);
            named_bar(bar_id, GROUP);
            {
                const int r8 = t & 7;
                const uint32_t nb = Nst + (t >> 3) * 256, bq = bfin + (t >> 3) * 32;
                const float4 b0 = lds4(bq), b1 = lds4(bq + 16);
                const float bb[NB] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                float xt = 0.0f;
#pragma unroll
                for (int jj = 0; jj < NB; ++jj) {
                    const float4 n0 = lds4(nb + jj * 32), n1 = lds4(nb + jj * 32 + 16);
                    const float nr[NB] = {n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, n1.z, n1.w};
                    float y = 0.0f;
#pragma unroll
                    for (int kk = 0; kk <= jj; ++kk) y = fmaf(nr[kk], bb[kk], y);
                    float nsel = 0.0f;  // N[jj][r8] (zero above the diagonal)
#pragma unroll
                    for (int kk = 0; kk <= jj; ++kk) nsel = (kk == r8) ? nr[kk] : nsel;
                    xt = fmaf(nsel, y, xt);
                }
                xout[t] = t < f8 ? xt * inv_s2 : 0.0f;  // N was stored as S N; padding columns of the whitened solution are 0
            }
            named_bar(bar_id, GROUP);  // Nst / bfin are rewritten by the next row
            if (prof) t_back += clock64() - tt;
        }
        if (prof) {
            p.prof[16] = clock64() - t_start; p.prof[17] = t_accfull; p.prof[18] = t_fact; p.prof[19] = t_back;
            p.prof[22] = my_rows; p.prof[24] = ph_wait; p.prof[25] = ph_ld; p.prof[26] = ph_own; p.prof[28] = ph_p;
            p.prof[31] = ph_issue; p.prof[32] = cg_rows; p.prof[33] = cg_products;
        }
    }
    // =============================== TEARDOWN ===============================
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// f <= 256: every width goes through the whitened pipeline (factors padded to 128 or 256 columns). Rows with at
// most tc_dual_max_entries() stored entries take the dual kernel at any width; longer rows take the primal kernel
// of this file when f <= 128 and the 256-wide one (half_step_tc256.cu) above that. Biases are a shifted weight
// (wmf_model.py:343); only rows with a negative weight go to the CUDA-core LU kernel.
bool tc_half_step_supported(int f, int bias) { return f >= 1 && f <= 256 && (!bias || f >= 2); }

// Workspace (bytes from a 256-aligned base):
//   [0, 1024)   header: [1] flags (1 unused, 2 failed pivot, 8 G not positive definite), [2] max y~^2 (float bits),
//               [4] total slots, [5] split rows, [6] partial slots, [7] extra slots, [8] fix-up rows, [9] end of the
//               primal rows' slots, [10] 0x7fffffff - first dual slot, [11] end of the dual rows' slots, [12] nonzero when the
//               conjugate gradients of some row did not converge (factorised instead), [13] packs of the dual kernel,
//               [14 .. 17] dual rows of 1 ... 4 slices; [256, 768) profile
//   tables      primal row table + split table (32 B per slot), dual row table (16 B per slot), dual-row counts per
//               chunk of PACK_CHUNK slots (16 B), split-row counters, fix-up list (4 B per row), dual pack table (64 B per
//               row: a pack holds at least one row, and a schedule names a row at most once, as the fix-up list assumes)
//   whitening   double scratch of the Cholesky, the two FP x FP multipliers, Y~ (cols x FP), X' (rows x FP)
//   simt        the CUDA-core kernel's own workspace (fix-up rows)
//   parts       partial-Gram scratch for the segments of split rows: whatever is left
struct TcLayout {
    int64_t cap_slots, max_parts;
    int64_t pack_chunks;
    size_t off_tab, off_seg, off_dtab, off_pcnt, off_cnt, off_fix, zero_end, off_ptab, off_chol, off_mw, off_mu, off_eye,
        off_yt, off_xp, off_simt, off_parts, total;
};
static int tc_fp(int f) { return f <= 128 ? 128 : 256; }
static size_t part_floats(int f) { return f <= F ? PART_FLOATS : tc256_part_floats(); }  // a parked segment: matrix + rhs
static TcLayout tc_layout(int64_t sched_slots, int64_t rows, int64_t cols, int f, int64_t parts) {
    TcLayout L;
    const size_t FP = (size_t)tc_fp(f);
    L.max_parts = parts < 2 ? 0 : parts;
    L.cap_slots = sched_slots + L.max_parts;
    L.off_tab = WS_TABLES;
    L.off_seg = L.off_tab + 16 * (size_t)L.cap_slots;
    L.off_dtab = L.off_seg + 16 * (size_t)L.cap_slots;
    L.pack_chunks = (sched_slots + PACK_CHUNK - 1) / PACK_CHUNK;
    L.off_pcnt = L.off_dtab + 16 * (size_t)sched_slots;
    L.off_cnt = L.off_pcnt + 16 * (size_t)L.pack_chunks;
    L.off_fix = align_up(L.off_cnt + 4 * (size_t)(L.max_parts / 2 + 1), 256);
    L.zero_end = L.off_fix;  // header, tables and counters are cleared per call; the list is bounded by its counter
    L.off_ptab = align_up(L.off_fix + 4 * (size_t)(rows + 1), 256);   // written in full up to its pack count
    L.off_chol = align_up(L.off_ptab + 64 * (size_t)(rows < sched_slots ? rows : sched_slots), 256);
    L.off_mw = L.off_chol + whiten_scratch_bytes(f);
    L.off_mu = L.off_mw + FP * FP * sizeof(float);
    L.off_eye = L.off_mu + FP * FP * sizeof(float);           // f x f identity: the whitened G of the fix-up kernel
    L.off_yt = L.off_eye + FP * FP * sizeof(float);
    L.off_xp = align_up(L.off_yt + (size_t)cols * FP * sizeof(float), 256);
    L.off_simt = align_up(L.off_xp + (size_t)rows * FP * sizeof(float), 256);
    L.off_parts = align_up(L.off_simt + simt_half_step_workspace_bytes(f), 256);
    L.total = L.off_parts + (size_t)L.max_parts * part_floats(f) * sizeof(float);
    return L;
}
size_t tc_half_step_workspace_bytes(int64_t rows, int64_t cols, int f, int, int64_t segments) {
    if (segments < 0) segments = rows >= 1024 ? DEFAULT_PARTS : 128;
    return tc_layout(2 * rows + 4096 + 1024, rows, cols, f, segments + 2).total;
}

int wmf_tc_split_length() { return split_len(); }

int tc_half_step(const HalfStepParams& in, void* ws, size_t ws_bytes, cudaStream_t st) {
    const int sms = sm_count();
    int grid = sms;
    if ((int64_t)grid > in.sched_len) grid = (int)in.sched_len;
    const int64_t extra_slot0 = (in.sched_len + grid - 1) / grid * grid;
    const int FP = tc_fp(in.f);
    const size_t need = tc_layout(extra_slot0, in.rows, in.cols, in.f, 0).total;
    if (ws == nullptr || ws_bytes < need) {
        set_error("wmf_als_half_step(tcgen05): workspace %zu < %zu (schedule of %lld slots, %lld x %lld, f = %d)", ws_bytes,
                  need, (long long)in.sched_len, (long long)in.rows, (long long)in.cols, in.f);
        return WMF_ERR_WORKSPACE;
    }
    // whatever is left after the fixed regions is scratch for the segments of split rows (each needs 34 bytes of tables too)
    int64_t max_parts = (int64_t)((ws_bytes - need) / (part_floats(in.f) * sizeof(float) + 34 + 8)) - 4;
    if (max_parts < 2) max_parts = 0;
    if (max_parts > (1ll << 24)) max_parts = 1ll << 24;
    const TcLayout L = tc_layout(extra_slot0, in.rows, in.cols, in.f, max_parts);
    if (L.total > ws_bytes) { set_error("wmf_als_half_step(tcgen05): internal workspace layout error"); return WMF_ERR_WORKSPACE; }
    max_parts = L.max_parts;
    char* base = reinterpret_cast<char*>(ws);
    uint32_t* hdr_u = reinterpret_cast<uint32_t*>(base);
    int* flags = reinterpret_cast<int*>(base) + 1;
    int4* tab = reinterpret_cast<int4*>(base + L.off_tab);
    int4* segtab = reinterpret_cast<int4*>(base + L.off_seg);
    int4* dtab = reinterpret_cast<int4*>(base + L.off_dtab);
    int* counters = reinterpret_cast<int*>(base + L.off_cnt);
    float* Mw = reinterpret_cast<float*>(base + L.off_mw);
    float* Mu = reinterpret_cast<float*>(base + L.off_mu);
    float* Yt = reinterpret_cast<float*>(base + L.off_yt);
    float* Xp = reinterpret_cast<float*>(base + L.off_xp);
    float* parts = reinterpret_cast<float*>(base + L.off_parts);
    WMF_CUDA(cudaMemsetAsync(ws, 0, L.zero_end, st));                       // header, empty tables, counters
    WMF_CUDA(cudaMemsetAsync(base + L.off_simt, 0, 256, st));               // the CUDA-core kernel's row counter
    // ---- whiten: L = chol(G), Y~ = Y L^-T (zero padded to FP columns), running max of y~^2 -> hdr[2]
    int rc = chol_whiten(in.G, in.f, FP, base + L.off_chol, Mw, Mu, reinterpret_cast<float*>(base + L.off_eye), flags, st);
    if (rc) return rc;
    rc = right_multiply(in.Y, in.cols, in.ldy, in.f, in.bias, Mw, FP, Yt, FP, FP, hdr_u + 2, st);
    if (rc) return rc;
    HalfStepParams p = in;
    p.Yraw = in.Y; p.ldraw = in.ldy;
    p.Y = Yt; p.ldy = FP;
    p.X = Xp; p.ldx = FP;
    p.FP = FP;
    p.f8 = (in.f + 7) / 8 * 8;
    p.f16 = (in.f + 15) / 16 * 16;
    p.fix_list = reinterpret_cast<int*>(base + L.off_fix);
    p.fix_count = reinterpret_cast<int*>(hdr_u + 8);
    // wider than 128 features one row at a time fits the tensor memory of an SM (half_step_tc256.cu): the dual kernel
    // (four n x n systems in flight) takes everything it can hold, n <= 128
    p.nd_max = dual_enabled() ? (FP > F ? 128 : tc_dual_max_entries()) : 0;
    p.prof = profile_enabled() ? reinterpret_cast<long long*>(base + WS_PROF) : nullptr;
    const int primal_ok = 1;   // 128-wide kernel of this file, or the 256-wide one (half_step_tc256.cu)
    uint32_t* pcnt = reinterpret_cast<uint32_t*>(base + L.off_pcnt);
    tc_prep_rows_kernel<<<(unsigned)((in.sched_len + 7) / 8), 256, 0, st>>>(p, tab, segtab, dtab, pcnt, hdr_u, extra_slot0,
                                                                            (int)max_parts, (int)max_parts, split_len(),
                                                                            primal_ok);
    WMF_LAUNCH_CHECK("tc_prep_rows_kernel");
    const int pack_chunks = (int)((in.sched_len + PACK_CHUNK - 1) / PACK_CHUNK);
    tc_finish_prep_kernel<<<1, 1024, 0, st>>>(hdr_u, extra_slot0, (int)max_parts, reinterpret_cast<uint4*>(pcnt), pack_chunks);
    WMF_LAUNCH_CHECK("tc_finish_prep_kernel");
    if (p.nd_max > 0) {
        int4* ptab = reinterpret_cast<int4*>(base + L.off_ptab);
        tc_pack_dual_kernel<<<(unsigned)pack_chunks, PACK_CHUNK, 0, st>>>(dtab, reinterpret_cast<const uint4*>(pcnt), hdr_u,
                                                                          ptab, in.sched_len);
        WMF_LAUNCH_CHECK("tc_pack_dual_kernel");
        rc = tc_dual_launch(p, ptab, hdr_u, grid, st);
        if (rc) return rc;
    }
    if (in.f > F) {
        rc = tc256_launch(p, tab, segtab, parts, counters, hdr_u, extra_slot0, flags, grid, st);
        if (rc) return rc;
    } else {
        // TMA descriptor of the whitened factors Y~ [cols x 128] for the row gathers (tile::gather4: one 512-byte row
        // per box, four row indices per instruction; rows past `cols` read as zeros)
        CUtensorMap ymap;
        {
            const cuuint64_t gdim[2] = {(cuuint64_t)F, (cuuint64_t)(in.cols > 0 ? in.cols : 1)};
            const cuuint64_t gstride[1] = {(cuuint64_t)F * sizeof(float)};
            const cuuint32_t box[2] = {(cuuint32_t)F, 1u}, estr[2] = {1u, 1u};
            // the driver entry point is looked up at run time: the library must load on a machine without libcuda
            // (the build check runs on a CPU-only box)
            static const PFN_cuTensorMapEncodeTiled_v12000 encode = [] {
                void* fn = nullptr;
                cudaDriverEntryPointQueryResult q;
                if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess ||
                    q != cudaDriverEntryPointSuccess)
                    fn = nullptr;
                return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
            }();
            if (encode == nullptr) { set_error("wmf_als_half_step(tcgen05): cuTensorMapEncodeTiled is not available in this driver"); return WMF_ERR_CUDA; }
            const CUresult cr = encode(&ymap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, Yt, gdim, gstride, box, estr,
                                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                       CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (cr != CUDA_SUCCESS) { set_error("wmf_als_half_step(tcgen05): cuTensorMapEncodeTiled failed (%d)", (int)cr); return WMF_ERR_CUDA; }
        }
        // the attribute is per device: set it on every call (a process may drive several GPUs)
        if (p.prof) {
#ifdef WMF_TC_PROFILE_BUILD
            WMF_CUDA(cudaFuncSetAttribute(als_half_step_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
            als_half_step_tc_kernel<true><<<grid, THREADS, SMEM_BYTES, st>>>(ymap, p, tab, segtab, parts, counters, hdr_u, extra_slot0, flags);
#endif
        } else {
            WMF_CUDA(cudaFuncSetAttribute(als_half_step_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
            als_half_step_tc_kernel<false><<<grid, THREADS, SMEM_BYTES, st>>>(ymap, p, tab, segtab, parts, counters, hdr_u, extra_slot0, flags);
        }
        WMF_LAUNCH_CHECK("als_half_step_tc_kernel");
    }
    // ---- fix-up: the CUDA-core LU kernel solves the listed rows, in the whitened variables as well (same
    // conditioning as the tensor-core rows): Y~, G = I, weights shifted by the original bias column
    HalfStepParams fix = in;
    fix.Y = Yt; fix.ldy = FP;
    fix.Yraw = in.Y; fix.ldraw = in.ldy;
    fix.G = reinterpret_cast<const float*>(base + L.off_eye);
    fix.X = Xp; fix.ldx = FP;
    fix.row_order = p.fix_list;
    fix.sched_len = in.rows;
    fix.sched_len_dev = p.fix_count;
    rc = simt_half_step(fix, base + L.off_simt, simt_half_step_workspace_bytes(in.f), st);
    if (rc) return rc;
    // ---- unwhiten: X = X' L^-1
    return right_multiply(Xp, in.rows, FP, in.f, 0, Mu, FP, in.X, in.ldx, in.f, nullptr, st);
}

}  // namespace wmf
