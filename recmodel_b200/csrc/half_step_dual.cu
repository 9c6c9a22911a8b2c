// K2 (tcgen05, dual form): ALS rows with few stored entries, any factor width up to 256, with or without biases.
// Replaces the per-row loop of recompute_factors / recompute_factors_bias (wmf_model.py:220-239, :337-350) for
// the rows tc_prep_rows_kernel routes here (0 < n <= ND_MAX entries, all weights > 0).
//
// With whitened factors y~ = L^-1 y (G = L L^T, whiten.cu) a row's system is (I + W^T W) x' = W^T c with
// W = diag(sqrt d) Y~_r  (n x f) and c_j = (d_j + 1) / sqrt(d_j). Push-through:  x' = W^T u,  (I + W W^T) u = c,
// an n x n system instead of f x f: a user with 40 entries pays 5 Gauss-Jordan steps instead of 16 (f = 128) or 32
// (f = 256), and the system matrix has its spectrum in [1, ~10] whatever the factors look like.
//
// Packs: a system of n entries takes dual_slices(n) = ceil(n16 / 32) 32-lane slices of a group's 128 TMEM lanes, and
// up to four systems share them on the block diagonal, lanes and columns at the same offset (tc_pack_dual_kernel
// builds the packs: {4}, {3,1}, {2,2}, {2,1,1}, {1,1,1,1} slices, with fewer 1-slice partners where they run out).
// TMEM lane quarter q is read only by warps with warp % 4 == q, which sit on SM sub-partition q: one system per group
// would leave a short row on one scheduler and three warps idle. A row's arithmetic does not depend on its pack or
// place in it.
//
//   Gram    W W^T on the tensor cores: the gathered factor rows ARE the K-major operand rows (K = features), so a
//           gather warp loads a row with one coalesced 512-byte read, scales by S sqrt(d_j), splits to FP16 hi/lo
//           and stores 8-byte pieces into the 128-byte-swizzled tiles: no transposition through shared memory.
//           One operand stage = 64 features x 128 tile rows (hi + lo, 32 KB); a pack takes f_pad / 64 stages; three
//           tcgen05.mma (kind::f16, M = N = 128, K = 16) per 16 features, fp32 accumulation in TMEM.
//   Solve   conjugate gradients (cg_solve.cuh) per system on its own warps; the systems that do not converge get
//           the block Gauss-Jordan in TMEM, 8 columns per step, exactly the scheme of half_step_tc.cu (pivot block
//           factored by one warp, rank-8 update as three kind::tf32 MMAs).
//   x'      = sum_j u_j sqrt(d_j) y~_j: thread m sums feature m over the row's entries (coalesced re-reads of the
//           factor rows the gather warps have just pulled through L2), written to the whitened solution X'.
//
// Roles as in the primal kernel: warps 0-15 four solver groups (one 128-column accumulator each), warps 16-23 gather,
// warp 24 MMA issue. One persistent CTA per SM walks the packs k * gridDim + blockIdx of the pack table.
#include <stdlib.h>
#include "tc_common.cuh"
#include "half_step.cuh"
#include "factor8.cuh"
#include "cg_solve.cuh"

namespace wmf {

namespace dual {

using namespace tc;

constexpr int ND_MAX = 96;            // longest row taken here (rounded up to 16 it must fit 128 TMEM lanes)
constexpr int NST = 5;                // operand stages
constexpr int TILE_BYTES = 128 * 128; // 128 entries x 64 fp16 features
constexpr int PAIR_BYTES = 2 * TILE_BYTES;
constexpr int NB = 8;
constexpr int NGROUP = 4, GROUP = 128;
#ifndef WMF_DUAL_NGATHER
#define WMF_DUAL_NGATHER 8
#endif
constexpr int NGATHER = WMF_DUAL_NGATHER;   // gather warps
static_assert(NGATHER >= 4 && 128 % NGATHER == 0, "a gather lane holds one tile row");
constexpr int SOLVER_WARP0 = 0, GATHER_WARP0 = NGROUP * 4, MMA_WARP = GATHER_WARP0 + NGATHER;
constexpr int THREADS = (MMA_WARP + 1) * 32;  // 800
constexpr uint32_t TMEM_COLS = 512;
constexpr int ACC_COLS = 128;
// named barriers 1 .. NGROUP: a whole solver group; CG_BAR0 + 2 g + s / 2: the warps of its system of more than one
// slice that starts at slice s (0 or 2); one-slice systems need none
constexpr int CG_BAR0 = 1 + NGROUP;
static_assert(CG_BAR0 + 2 * NGROUP <= 16, "named barriers");

constexpr int PANEL_TILE_BYTES = 128 * NB * 4;
constexpr int G_OFF_TILEH = 0;
constexpr int G_OFF_TILEL = G_OFF_TILEH + PANEL_TILE_BYTES;
constexpr int G_OFF_NINV = G_OFF_TILEL + PANEL_TILE_BYTES;
constexpr int G_OFF_ZB = G_OFF_NINV + 16 * NB * NB * 4;
constexpr int G_OFF_DBLK = G_OFF_ZB + 16 * NB * 4;
constexpr int G_OFF_BFIN = G_OFF_DBLK + (NB * NB + 2 * NB) * 4;
constexpr int G_OFF_PAIRS = ((G_OFF_BFIN + 128 * 4 + 15) / 16) * 16;   // 128 x (coefficient, factor row)
constexpr int G_OFF_CGOK = G_OFF_PAIRS + 128 * 8;                         // 2 x 4 slices: converged?
constexpr int GROUP_BYTES = ((G_OFF_CGOK + 2 * 16 + 127) / 128) * 128;

constexpr int OFF_STAGES = 0;
constexpr int OFF_GROUPS = OFF_STAGES + NST * PAIR_BYTES;
constexpr int OFF_BARS = OFF_GROUPS + NGROUP * GROUP_BYTES;
constexpr int NBARS = 2 * NST + 3 * NGROUP;
constexpr int OFF_TMEM_PTR = OFF_BARS + NBARS * 8;
constexpr int SMEM_BYTES = OFF_TMEM_PTR + 16 + 1024;
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(ND_MAX % 16 == 0 && ND_MAX <= 128, "dual rows must fit the TMEM lanes");  // the kernel itself takes any n <= 128

__global__ void __launch_bounds__(THREADS, 1)
als_half_step_dual_kernel(HalfStepParams p, const int4* __restrict__ ptab, const uint32_t* __restrict__ hdr_u,
                          int* __restrict__ flags) {
    extern __shared__ uint8_t smem_raw[];
    // packs [0, hdr[13]) of the pack table (tc_pack_dual_kernel); none: nothing to set up
    const int npacks = (int)hdr_u[13];
    if (npacks == 0) return;
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = smem_base + OFF_BARS;
    auto bar_full = [&](int s) { return bars + 8u * s; };
    auto bar_empty = [&](int s) { return bars + 8u * (NST + s); };
    auto bar_acc_full = [&](int g) { return bars + 8u * (2 * NST + g); };
    auto bar_acc_empty = [&](int g) { return bars + 8u * (2 * NST + NGROUP + g); };
    auto bar_panel = [&](int g) { return bars + 8u * (2 * NST + 2 * NGROUP + g); };

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int FP = p.FP, KCH = FP >> 6, PASSES = FP >> 7;

    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(bar_full(s), NGATHER); mbar_init(bar_empty(s), 1); }
        for (int g = 0; g < NGROUP; ++g) {
            mbar_init(bar_acc_full(g), 1);
            mbar_init(bar_acc_empty(g), GROUP);
            mbar_init(bar_panel(g), 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // operand rows outside every system of a pack are read by the MMA (they only reach TMEM lanes and columns nobody
    // uses): start from finite values
    for (uint32_t o = (uint32_t)tid * 16u; o < (uint32_t)(NST * PAIR_BYTES); o += THREADS * 16u)
        sts4u(smem_base + OFF_STAGES + o, 0u, 0u, 0u, 0u);
    fence_async_smem();
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

    const int ts = (int)gridDim.x;
    const int npk = (npacks - (int)blockIdx.x + ts - 1) / ts;   // this CTA's packs: k * ts + blockIdx
    auto pack_ent = [&](int k, int slice) -> int4 {               // entry of the system covering `slice` of pack k
        int4 v = make_int4(-1, 0, 0, 0);
        if (k < npk) v = __ldg(ptab + ((int64_t)k * ts + (int64_t)blockIdx.x) * 4 + slice);
        return v;
    };

    if (warp >= GATHER_WARP0 && warp < MMA_WARP) {
        // =============================== GATHER ===============================
        const int w = warp - GATHER_WARP0;
        const int csel = lane >> 4;                 // which 64-feature chunk of a 128-feature pass this lane feeds
        const uint32_t q = (uint32_t)(lane & 15) >> 1, half8 = (uint32_t)(lane & 1) * 8u;
        uint32_t gsi = 0;                           // stages consumed so far by this CTA
        // The warp writes the tile rows j = w, w + NGATHER, ... of a pack: lane l holds row j = w + NGATHER l, which is
        // entry j - 32 s of the system whose slices start at s, a zero padding row up to that system's n16, or no
        // row of any system (nothing written: it only reaches off-diagonal blocks). Indices and weights are fetched one
        // pack ahead (nothing may depend on those loads in the step that issues them), and the factor rows are read
        // four entries at a time with the next four already in flight: every global-load latency of a row used to be
        // exposed once per row / per four entries, which made the gather the critical path of this kernel.
        constexpr int RPW = 128 / NGATHER;        // tile rows per warp
        const int my_slice = lane < RPW ? (w + NGATHER * lane) >> 5 : 0;
        struct Pre { int idx; float d; int sexp; };   // idx -1: zero padding, -2: no row
        auto fetch = [&](const int4 v) -> Pre {
            Pre o{-2, 0.0f, 0};
            if (lane < RPW && v.y > 0) {
                const RowEnt r = unpack_ent(v, 0);
                const int j = w + NGATHER * lane - 32 * pack_first_slice(v);
                if (j < r.n) {
                    o.idx = __ldg(p.indices + r.lo + j);
                    o.d = __ldg(p.data + r.lo + j);
                    o.sexp = r.sexp;
                } else if (j < ((r.n + 15) & ~15)) {
                    o.idx = -1;
                }
            }
            return o;
        };
        int4 cur = pack_ent(0, my_slice), nxt = pack_ent(1, my_slice);
        Pre pc = fetch(cur);
        for (int k = 0; k < npk; ++k) {
            const Pre pe = pc;
            cur = nxt;
            nxt = pack_ent(k + 2, my_slice);
            pc = fetch(cur);
            const int my_idx = pe.idx;
            float my_s = 0.0f;
            if (my_idx >= 0) {
                float d = pe.d;
                if (p.bias) d = __fsub_rn(d, __ldg(p.Yraw + (int64_t)my_idx * p.ldraw));  // wmf_model.py:343
                my_s = exp2f((float)pe.sexp) * sqrtf(d);
            }
            for (int c = 0; c < KCH; ++c) {
                const uint32_t gs = gsi + (uint32_t)c;
                mbar_wait(bar_empty(gs % NST), ((gs / NST) & 1u) ^ 1u);
            }
            for (int ps = 0; ps < PASSES; ++ps) {
                const uint32_t sb = smem_base + OFF_STAGES + ((gsi + (uint32_t)(ps * 2 + csel)) % NST) * PAIR_BYTES;
                const float* ybase = p.Y + ps * 128 + lane * 4;
                auto load4 = [&](int e0, float4 (&v)[4]) {   // e0 is warp-uniform
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const int idx = __shfl_sync(0xffffffffu, my_idx, (e0 + b) & 31);
                        v[b] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (idx >= 0) v[b] = __ldg(reinterpret_cast<const float4*>(ybase + (int64_t)idx * FP));
                    }
                };
                auto store4 = [&](int e0, const float4 (&v)[4]) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const float ss = __shfl_sync(0xffffffffu, my_s, (e0 + b) & 31);
                        const int idx = __shfl_sync(0xffffffffu, my_idx, (e0 + b) & 31);
                        if (idx == -2) continue;   // no row of any system: nothing to write
                        const uint32_t j = (uint32_t)(w + NGATHER * (e0 + b));
                        const uint32_t roff = (j >> 3) * 1024u + (j & 7u) * 128u + (((q ^ (j & 7u))) << 4) + half8;
                        const float z0 = ss * v[b].x, z1 = ss * v[b].y, z2 = ss * v[b].z, z3 = ss * v[b].w;
                        const __half2 h01 = __floats2half2_rn(z0, z1), h23 = __floats2half2_rn(z2, z3);
                        const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                        const __half2 l01 = __floats2half2_rn(z0 - f01.x, z1 - f01.y), l23 = __floats2half2_rn(z2 - f23.x, z3 - f23.y);
                        sts2u(sb + roff, h2_bits(h01), h2_bits(h23));
                        sts2u(sb + TILE_BYTES + roff, h2_bits(l01), h2_bits(l23));
                    }
                };
                float4 va[4], vb[4];
                load4(0, va);
                for (int e0 = 0; e0 < RPW; e0 += 8) {
                    load4(e0 + 4, vb);
                    store4(e0, va);
                    if (e0 + 8 < RPW) load4(e0 + 8, va);
                    store4(e0 + 4, vb);
                }
            }
            fence_async_smem();   // generic-proxy stores -> visible to the tensor core (async proxy)
            __syncwarp();
            if (lane == 0)
                for (int c = 0; c < KCH; ++c) mbar_arrive(bar_full((gsi + (uint32_t)c) % NST));
            gsi += (uint32_t)KCH;
        }
    } else if (warp == MMA_WARP) {
        // =============================== GRAM MMA ISSUE ===============================
        // warp-uniform loop, one elected lane issues (see elect_one()). One M = N = 128 chain per pack over the whole
        // tile: the diagonal blocks are the pack's systems, the off-diagonal blocks are never read.
        {
            uint32_t gsi = 0;
            const uint32_t idesc = IDESC_F16_M128 | ((uint32_t)(ACC_COLS >> 3) << 17);
            for (int k = 0; k < npk; ++k) {
                const int g = k % NGROUP;
                mbar_wait(bar_acc_empty(g), ((k / NGROUP) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(g * ACC_COLS);
                uint32_t accumulate = 0;
                for (int c = 0; c < KCH; ++c, ++gsi) {
                    const uint32_t s = gsi % NST;
                    mbar_wait(bar_full(s), (gsi / NST) & 1u);
                    tc_fence_after();
                    const uint32_t tile = smem_base + OFF_STAGES + s * PAIR_BYTES;
                    const uint64_t dh = umma_desc(tile), dl = umma_desc(tile + TILE_BYTES);
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {   // 16 fp16 features = 32 B along K inside the 128-B swizzle row
                            const uint64_t hk = dh + (uint64_t)(kk * 2), lk = dl + (uint64_t)(kk * 2);
                            umma_f16(d_tmem, hk, hk, idesc, kk == 0 ? accumulate : 1u);  // wh wh^T
                            umma_f16(d_tmem, hk, lk, idesc, 1u);          // wh wl^T
                            umma_f16(d_tmem, lk, hk, idesc, 1u);          // wl wh^T
                        }
                        tc_commit(bar_empty(s));
                    }
                    __syncwarp();
                    accumulate = 1;
                }
                if (elect_one()) tc_commit(bar_acc_full(g));
                __syncwarp();
            }
        }
    } else {
        // =============================== SOLVE (the pack's n x n matrices resident in TMEM) ===============================
        const int g = (warp - SOLVER_WARP0) >> 2;
        const int qw = warp & 3;        // TMEM lane quarter this warp may access = the pack slice it serves
        const int tl = qw * 32 + lane;  // TMEM lane of this thread: row tl - 32 s of the system whose slices start at s
        const int bar_id = 1 + g;
        const int ISSUE_T = 32 * g;  // thread of the group that issues its rank-8 update MMAs
        const uint32_t gs = smem_base + OFF_GROUPS + g * GROUP_BYTES;
        const uint32_t tileH = gs + G_OFF_TILEH, tileL = gs + G_OFF_TILEL;
        const uint32_t Nst = gs + G_OFF_NINV, zst = gs + G_OFF_ZB, Dblk = gs + G_OFF_DBLK, bfin = gs + G_OFF_BFIN;
        const uint32_t pairs = gs + G_OFF_PAIRS, cg_ok = gs + G_OFF_CGOK;
        const uint32_t t_lane = tmem_base + ((uint32_t)(qw * 32) << 16) + (uint32_t)(g * ACC_COLS);
        const uint32_t d_tmem = tmem_base + (uint32_t)(g * ACC_COLS);
        const uint64_t descH = umma_desc_panel(tileH), descL = umma_desc_panel(tileL);
        uint32_t panel_n = 0;
#ifdef WMF_TC_PROFILE_BUILD
        const bool prof_g = p.prof != nullptr && blockIdx.x == 0 && g == 0;   // every system of this group: rows, products, entries
        const bool prof = prof_g && tl == 0;                                  // phase clocks
        long long pf_t0 = prof ? clock64() : 0, pf_acc = 0, pf_cg = 0, pf_xp = 0, pf_a = 0, pf_b = 0;
#endif
        int4 nxt = pack_ent(g, qw);
        for (int k = g; k < npk; k += NGROUP) {
            const int4 v = nxt;
            const uint32_t ph = (uint32_t)(k / NGROUP) & 1u;
            // this thread's system (n = 0: no system covers this warp's slice) and its entry t of it: weight, factor
            // row, right-hand side c_t = (d_t + 1) / sqrt(d_t)
            const RowEnt e = unpack_ent(v, 0);
            const int s0 = pack_first_slice(v);
            const bool active = e.n > 0;
            const int n = e.n, n16 = (n + 15) & ~15, nsl = dual_slices(n);
            const int t = tl - 32 * s0;
            const uint32_t t_row = t_lane + (uint32_t)(32 * s0);
            const float inv_s = exp2f((float)-e.sexp), inv_s2 = inv_s * inv_s;
            int my_idx = 0;
            float sq = 0.0f, bt = 0.0f;
            if (t < n) {
                my_idx = __ldg(p.indices + e.lo + t);
                float d = __ldg(p.data + e.lo + t);
                if (p.bias) d = __fsub_rn(d, __ldg(p.Yraw + (int64_t)my_idx * p.ldraw));
                sq = sqrtf(d);
                bt = __fdiv_rn(__fadd_rn(d, 1.0f), sq);
            }
#ifdef WMF_TC_PROFILE_BUILD
            if (prof) pf_a = clock64();
#endif
            mbar_wait(bar_acc_full(g), ph);
#ifdef WMF_TC_PROFILE_BUILD
            if (prof) { pf_b = clock64(); pf_acc += pf_b - pf_a; }
#endif
            tc_fence_after();
            // ---- default solver: conjugate gradients against the matrix in tensor memory (cg_solve.cuh), each system
            // on its own warps, vector / reduction scratch and named barrier; the block Gauss-Jordan below takes the
            // systems that have not converged within p.cg_maxit products
            float coef = 0.0f, xc = 0.0f;
            int products = -1;
            if (active && p.cg_maxit > 0) {
                products = cg_solve(t_row, t, n16, bt, inv_s2, bfin + 128u * (uint32_t)s0, Dblk + 64u * (uint32_t)s0, qw - s0,
                                    nsl, CG_BAR0 + 2 * g + (s0 >> 1), nsl * 32, p.cg_maxit, xc,
#ifdef WMF_TC_PROFILE_BUILD
                                    prof ? p.prof + 52 : nullptr
#else
                                    nullptr
#endif
                                    );
#ifdef WMF_TC_PROFILE_BUILD
                if (prof_g && t == 0) {
                    atomicAdd(reinterpret_cast<unsigned long long*>(p.prof + 44), 1ull);
                    atomicAdd(reinterpret_cast<unsigned long long*>(p.prof + 45), (unsigned long long)(long long)products);
                    atomicAdd(reinterpret_cast<unsigned long long*>(p.prof + 46), (unsigned long long)n);
                }
#endif
            }
            const uint32_t ok = cg_ok + ph * 16u;   // alternates between this group's consecutive packs
            if (lane == 0) sts1(ok + (uint32_t)qw * 4u, (!active || products >= 0) ? 1.0f : 0.0f);
            tc_fence_before();
            named_bar(bar_id, GROUP);
            const float4 okv = lds4(ok);
            nxt = pack_ent(k + NGROUP, qw);
            const uint32_t failed = (okv.x == 0.0f ? 1u : 0u) | (okv.y == 0.0f ? 2u : 0u) | (okv.z == 0.0f ? 4u : 0u) |
                                    (okv.w == 0.0f ? 8u : 0u);   // slices of the systems that have not converged
            if (t < n) coef = xc * sq;
            if (failed == 0) {
                mbar_arrive(bar_acc_empty(g));   // the Gram of this group's next pack may start
            } else {
                // header word 12: some row took the factorisation (a plain store: an atomicAdd at this point made the
                // whole kernel 50 % slower, measured A/B on one box, although it never executes on the bench workloads)
                if (p.cg_maxit > 0 && tl == 0) *reinterpret_cast<volatile int*>(flags + 11) = 1;
                tc_fence_after();
                // The systems that have not converged, one after the other with the whole group. The rank-8 updates of
                // one only change its own columns, which no other system of the pack reads.
#pragma unroll 1
                for (int sf = 0; sf < 4; ++sf) {
                    const int4 vf = pack_ent(k, sf);
                    if (!((failed >> sf) & 1u) || pack_first_slice(vf) != sf) continue;
                    const RowEnt ef = unpack_ent(vf, 0);
                    const int nf = ef.n, nf8 = (nf + 7) & ~7, nf16 = (nf + 15) & ~15;
                    const float Sf = exp2f((float)ef.sexp), inv_sf = exp2f((float)-ef.sexp);
                    const bool in = active && s0 == sf;   // this thread holds a row of that system
#pragma unroll 1
                    for (int c0 = 0; c0 < nf8; c0 += NB) {
                        if (c0 > 0) {  // the previous step's rank-8 update has landed in TMEM
                            if (in) { mbar_wait(bar_panel(g), panel_n & 1u); tc_fence_after(); }
                            ++panel_n;
                        }
                        float a[NB] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                        if (in) tmem_ld8(t_row + c0, a);
                        const int rel = in ? t - c0 : -1;
#pragma unroll
                        for (int i = 0; i < NB; ++i) a[i] = fmaf(a[i], inv_s2, rel == i ? 1.0f : 0.0f);  // I + W W^T
                        const uint32_t nd = Nst + (c0 >> 3) * 256, zd = zst + (c0 >> 3) * 32;
                        // The 8 threads that hold the pivot rows publish them; the serial 8x8 factor is run by warp g of
                        // group g, whatever warp the pivot rows live in: the four groups' serial chains then sit on four
                        // different warp schedulers (warp id mod 4).
                        if (rel >= 0 && rel < NB) {
                            sts4(Dblk + rel * 32, a[0], a[1], a[2], a[3]);
                            sts4(Dblk + rel * 32 + 16, a[4], a[5], a[6], a[7]);
                            sts1(Dblk + 256 + rel * 4, bt);
                        }
                        named_bar(bar_id, GROUP);
                        if (qw == g) {
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
                            const bool okf = factor8(d, bb, lane & 7, ncol, z);  // lane c holds column c of N = L^-1
                            if (lane < NB) {
#pragma unroll
                                for (int i = 0; i < NB; ++i) sts1(nd + i * 32 + lane * 4, Sf * ncol[i]);
                            }
                            if (lane == 0) {
                                sts4(zd, inv_sf * z[0], inv_sf * z[1], inv_sf * z[2], inv_sf * z[3]);
                                sts4(zd + 16, inv_sf * z[4], inv_sf * z[5], inv_sf * z[6], inv_sf * z[7]);
                                if (!okf) {  // spectrum >= 1: only a numerical accident gets here; the LU kernel redoes the row
                                    atomicOr(flags, 2);
                                    p.fix_list[atomicAdd(p.fix_count, 1)] = ef.row;
                                }
                            }
                        }
                        named_bar(bar_id, GROUP);
                        float P[NB] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                        if (in) {
#pragma unroll
                            for (int jj = 0; jj < NB; ++jj) {
                                const float4 n0 = lds4(nd + jj * 32);
                                float x = a[0] * n0.x;
                                if (jj >= 1) x = fmaf(a[1], n0.y, x);
                                if (jj >= 2) x = fmaf(a[2], n0.z, x);
                                if (jj >= 3) x = fmaf(a[3], n0.w, x);
                                if (jj >= 4) {
                                    const float4 n1 = lds4(nd + jj * 32 + 16);
                                    x = fmaf(a[4], n1.x, x);
                                    if (jj >= 5) x = fmaf(a[5], n1.y, x);
                                    if (jj >= 6) x = fmaf(a[6], n1.z, x);
                                    if (jj >= 7) x = fmaf(a[7], n1.w, x);
                                }
                                P[jj] = x;
                            }
                            if (qw - sf == (c0 >> 5)) {
                                const bool pivot = rel >= 0 && rel < NB;
#pragma unroll
                                for (int jj = 0; jj < NB; ++jj) P[jj] = pivot ? 0.0f : P[jj];
                            }
                            const float4 z0 = lds4(zd), z1 = lds4(zd + 16);
                            float u0 = P[0] * z0.x, u1 = P[1] * z0.y;
                            u0 = fmaf(P[2], z0.z, u0); u1 = fmaf(P[3], z0.w, u1);
                            u0 = fmaf(P[4], z1.x, u0); u1 = fmaf(P[5], z1.y, u1);
                            u0 = fmaf(P[6], z1.z, u0); u1 = fmaf(P[7], z1.w, u1);
                            bt -= u0 + u1;
                        }
                        if (c0 + NB < nf8) {
                            if (in) {
                                float lh[NB], ll[NB];
#pragma unroll
                                for (int jj = 0; jj < NB; ++jj) {
                                    lh[jj] = tf32_round(P[jj]);
                                    ll[jj] = P[jj] - lh[jj];
                                }
                                const uint32_t o = (uint32_t)((tl >> 3) * 256 + (tl & 7) * 16);   // panel row = TMEM lane
                                sts4(tileH + o, lh[0], lh[1], lh[2], lh[3]);
                                sts4(tileH + o + 128, lh[4], lh[5], lh[6], lh[7]);
                                sts4(tileL + o, ll[0], ll[1], ll[2], ll[3]);
                                sts4(tileL + o + 128, ll[4], ll[5], ll[6], ll[7]);
                                fence_async_smem();
                                tc_fence_before();
                            }
                            named_bar(bar_id, GROUP);
                            if (tl == ISSUE_T) {
                                tc_fence_after();
                                const uint32_t start = (uint32_t)((c0 + NB) >> 4) << 4;
                                const uint32_t col = (uint32_t)(32 * sf) + start;   // first column (and panel row) updated
                                const uint32_t idesc = IDESC_TF32_NEG_M128 | ((((uint32_t)nf16 - start) >> 3) << 17);
                                const uint64_t bH = descH + (uint64_t)(col * 2), bL = descL + (uint64_t)(col * 2);
                                umma_tf32(d_tmem + col, descH, bH, idesc, 1u);
                                umma_tf32(d_tmem + col, descH, bL, idesc, 1u);
                                umma_tf32(d_tmem + col, descL, bH, idesc, 1u);
                                tc_commit(bar_panel(g));
                            }
                        }
                    }
                    // ---- block diagonal now: u_blk = N^T (N b_blk); coefficient of factor row j: u_j sqrt(d_j) ----
                    if (in) sts1(bfin + t * 4, bt);
                    named_bar(bar_id, GROUP);
                    if (in) {
                        const int r8 = t & 7;
                        const uint32_t nb = Nst + (t >> 3) * 256, bq = bfin + (t >> 3) * 32;
                        const float4 b0 = lds4(bq), b1 = lds4(bq + 16);
                        const float bb[NB] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                        float xt = 0.0f;
                        if (t < nf8) {
#pragma unroll
                            for (int jj = 0; jj < NB; ++jj) {
                                const float4 n0 = lds4(nb + jj * 32), n1 = lds4(nb + jj * 32 + 16);
                                const float nr[NB] = {n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, n1.z, n1.w};
                                float y = 0.0f;
#pragma unroll
                                for (int kk = 0; kk <= jj; ++kk) y = fmaf(nr[kk], bb[kk], y);
                                float nsel = 0.0f;
#pragma unroll
                                for (int kk = 0; kk <= jj; ++kk) nsel = (kk == r8) ? nr[kk] : nsel;
                                xt = fmaf(nsel, y, xt);
                            }
                        }
                        coef = t < nf ? xt * inv_s2 * sq : 0.0f;   // N was stored as S N
                    }
                    named_bar(bar_id, GROUP);   // the scratch above is the next system's
                }
                tc_fence_before();
                mbar_arrive(bar_acc_empty(g));   // every system has read the accumulator: the next pack's Gram may start
            }
            asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(pairs + (uint32_t)tl * 8u), "r"(__float_as_uint(coef)),
                         "r"((uint32_t)my_idx) : "memory");
            named_bar(bar_id, GROUP);
#ifdef WMF_TC_PROFILE_BUILD
            if (prof) { pf_a = clock64(); pf_cg += pf_a - pf_b; }
#endif
            // ---- x'[m] = sum_j coef_j y~_j[m], for each system of the pack in turn with all four warps. Warp qw takes
            // the entries j = qw, qw + 4, ... (ascending) and lane l the features 4 l .. 4 l + 3 of a 128-feature pass:
            // one coalesced 512-byte read per factor row (the rows the gather warps have just pulled through L2), the
            // next four rows in flight while four are added; the four warps' partial sums meet in shared memory (the
            // panel tiles of the factorisation are free here) and thread tl adds them in warp order. A function of the
            // row alone, like everything else. ----
#pragma unroll 1
            for (int sm = 0; sm < 4; ++sm) {
                const int4 vm = pack_ent(k, sm);
                if (vm.y <= 0 || pack_first_slice(vm) != sm) continue;
                const int nm = vm.y;
                const uint32_t pm = pairs + (uint32_t)(32 * sm) * 8u;
                const uint32_t xpart = tileH;   // 4 warps x 256 floats
                for (int ps = 0; ps < PASSES; ++ps) {
                    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                    const float* yb = p.Y + ps * 128 + lane * 4;
                    auto load4 = [&](int j, float (&c)[4], float4 (&y)[4]) {   // j, nm are warp-uniform
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            c[b] = 0.0f;
                            y[b] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (j + 4 * b < nm) {
                                uint32_t cw, ci;
                                asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(cw), "=r"(ci) : "r"(pm + (uint32_t)(j + 4 * b) * 8u));
                                c[b] = __uint_as_float(cw);
                                y[b] = __ldg(reinterpret_cast<const float4*>(yb + (int64_t)ci * FP));
                            }
                        }
                    };
                    auto add4 = [&](const float (&c)[4], const float4 (&y)[4]) {
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            acc.x = fmaf(c[b], y[b].x, acc.x); acc.y = fmaf(c[b], y[b].y, acc.y);
                            acc.z = fmaf(c[b], y[b].z, acc.z); acc.w = fmaf(c[b], y[b].w, acc.w);
                        }
                    };
                    float ca[4], cb[4];
                    float4 ya[4], yv[4];
                    load4(qw, ca, ya);
                    for (int j = qw; j < nm; j += 32) {
                        if (j + 16 < nm) load4(j + 16, cb, yv);
                        add4(ca, ya);
                        if (j + 32 < nm) load4(j + 32, ca, ya);
                        if (j + 16 < nm) add4(cb, yv);
                    }
                    sts4(xpart + (uint32_t)((qw * 256 + ps * 128 + lane * 4) * 4), acc.x, acc.y, acc.z, acc.w);
                }
                named_bar(bar_id, GROUP);
                float* xout = p.X + (int64_t)vm.x * p.ldx;
                {
                    const uint32_t a = xpart + (uint32_t)tl * 4u;
                    xout[tl] = ((lds1(a) + lds1(a + 1024)) + lds1(a + 2048)) + lds1(a + 3072);
                    if (PASSES > 1) xout[128 + tl] = ((lds1(a + 512) + lds1(a + 1536)) + lds1(a + 2560)) + lds1(a + 3584);
                }
                named_bar(bar_id, GROUP);  // xpart is rewritten by the next system, pairs / Nst / bfin by the next pack
            }
#ifdef WMF_TC_PROFILE_BUILD
            if (prof) pf_xp += clock64() - pf_a;
#endif
        }
#ifdef WMF_TC_PROFILE_BUILD
        if (prof) { p.prof[40] = clock64() - pf_t0; p.prof[41] = pf_acc; p.prof[42] = pf_cg; p.prof[43] = pf_xp; }
#endif
    }
    // =============================== TEARDOWN ===============================
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

}  // namespace dual

// WMF_TC_DUAL_MAX=<entries> (multiple of 16, <= 128; read once) overrides the routing threshold for experiments
int tc_dual_max_entries() {
    static const int v = [] {
        const char* e = getenv("WMF_TC_DUAL_MAX");
        int x = e ? atoi(e) : dual::ND_MAX;
        if (x < 16 || x > 128) x = dual::ND_MAX;
        return x / 16 * 16;
    }();
    return v;
}

int tc_dual_launch(const HalfStepParams& p, const int4* ptab, const uint32_t* hdr_u, int grid, cudaStream_t st) {
    WMF_CUDA(cudaFuncSetAttribute(dual::als_half_step_dual_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  dual::SMEM_BYTES));
    int* flags = reinterpret_cast<int*>(p.fix_count) - 7;   // header word 1 (fix_count is word 8)
    dual::als_half_step_dual_kernel<<<grid, dual::THREADS, dual::SMEM_BYTES, st>>>(p, ptab, hdr_u, flags);
    WMF_LAUNCH_CHECK("als_half_step_dual_kernel");
    return WMF_OK;
}

}  // namespace wmf
