// PTX wrappers and small helpers shared by the tcgen05 half-step kernels (half_step_tc.cu: primal f x f systems,
// half_step_dual.cu: n x n systems of short rows). sm_100a only.
#pragma once
#include <cuda_fp16.h>
#include "common.cuh"

namespace wmf {
namespace tc {

// one 16-byte schedule-table entry per slot (see tc_prep_rows_kernel)
struct __align__(16) RowEnt {
    int32_t row;   // CSR row id, -1 = padding slot
    int32_t n;     // stored entries (0: nothing to do here: empty row, row of the other kernel, or fix-up row)
    int64_t lo;    // indptr[row] (48 bits when packed in the table)
    int32_t sexp;  // S = 2^sexp for this row (the table packs it into bits 16-23 of the last word)
    int32_t part;  // >= 0: this entry is a segment of a split row; index of its record in the split table (bit 31 flag)
};
__device__ __forceinline__ RowEnt unpack_ent(const int4 v, int slot) {
    RowEnt e;
    e.row = v.x; e.n = v.y; e.lo = ((int64_t)(uint32_t)v.z) | ((int64_t)(v.w & 0xFFFF) << 32);
    e.sexp = (int)(((uint32_t)v.w >> 16) & 0xFFu) - 64;
    e.part = (v.w < 0) ? slot : -1;
    return e;
}
// Dual kernel (half_step_dual.cu): an n-entry system takes dual_slices(n) 32-lane slices of its group's 128 TMEM
// lanes, and up to four systems share them on the block diagonal. The pack table holds four entries per pack, one per
// slice: the entry of the system covering that slice, with its first slice in bits 24-25 of the last word (n = 0: no
// system there).
__host__ __device__ __forceinline__ int dual_slices(int n) { return (n + 31) >> 5; }
__device__ __forceinline__ int pack_first_slice(const int4 v) { return (int)(((uint32_t)v.w >> 24) & 3u); }
// second table, one 16-byte record per segment of a split row
struct __align__(16) SegEnt {
    int32_t split_id;    // counter slot of the row
    int32_t nseg;        // segments of the row
    int32_t first_part;  // scratch slot of segment 0 (segments are consecutive)
    int32_t seg;         // this segment's index
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// try_wait with a suspend-time hint: the warp sleeps in hardware until the phase completes instead of
// re-polling every ~50 cycles (polling was 30 % of all issued instructions, ncu r01b).
// -DWMF_WATCHDOG (development builds only): a wait that does not complete within ~2 s traps instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
#ifdef WMF_WATCHDOG
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}" : "=r"(done) : "r"(bar), "r"(parity), "r"(0x989680u) : "memory");
        if (!done && spin > 400u) {
            printf("mbar_wait watchdog: block %d thread %d bar %u parity %u\n", blockIdx.x, threadIdx.x, bar, parity);
            __trap();
        }
    }
#else
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(bar), "r"(parity), "r"(0x989680u) : "memory");
#endif
}
// One lane of a converged warp (always the same one for a full mask). Around tcgen05.mma / tcgen05.commit it tells the
// compiler that exactly one thread issues them: `if (lane == 0)` makes it wrap every MMA in an ELECT / BRA.U.ANY loop
// and move each descriptor through R2UR (~85 cycles per MMA measured, scripts/probe/step_latency.cu), while a
// warp-uniform loop with the issue under elect.sync keeps descriptors in uniform registers.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
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
// MN-major ("transposed") operand, 128-byte swizzle: 64 contiguous M/N elements per swizzle row, 8 K rows per
// 1024-byte atom; LBO = bytes to the next 64 M/N elements, SBO = bytes to the next 8 K rows
// (cute::UMMA make_umma_desc<Major::MN>, verified by scripts/probe/mma_mn_major_probe.cu)
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (2ull << 61);
}
// K-major, no swizzle: 8-row x 16-byte core matrices; the two K-chunks of a row group are
// LBO = 128 B apart, consecutive 8-row groups SBO = 256 B apart (panel operand, K = 8 fp32).
__device__ __forceinline__ uint64_t umma_desc_panel(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) |
           (1ull << 46);
}
// cute::UMMA::InstrDescriptor: fp32 accumulate (bit 4), A/B formats at bits 7/10 (0 = F16, 2 = TF32),
// bit 13 negates A, N >> 3 at bit 17, M >> 4 at bit 24; K-major A and B.
constexpr uint32_t IDESC_F16_M128 = (1u << 4) | ((128u >> 4) << 24);                                            // N filled in at issue
constexpr uint32_t IDESC_MN_MAJOR_AB = (1u << 15) | (1u << 16);                                                 // A and B MN-major
constexpr uint32_t IDESC_TF32_NEG_M128 = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 13) | ((128u >> 4) << 24);  // N filled in at issue
#define TRI(i, j) ((i) * ((i) + 1) / 2 + (j))

__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

// A operand from tensor memory (128 lanes = M rows, K along the columns, two fp16 per 32-bit column), B from shared memory
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// round-to-nearest (ties away) to the 10-bit TF32 mantissa, done with integer ops
__device__ __forceinline__ float tf32_round(float x) {
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
                 "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                 "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                 "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_arrive(uint32_t bar) {  // arrive when this thread's copies have landed
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
// explicit shared-space accesses (generic ld/st on pointers derived from the aligned base cost an
// address-space check per access)
__device__ __forceinline__ float4 lds4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds1(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts4(uint32_t a, float x, float y, float z, float w) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ void sts4u(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void sts2u(uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void sts1(uint32_t a, float x) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(x) : "memory");
}
__device__ __forceinline__ void named_bar(int id, int count) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ uint32_t h2_bits(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }

// S = 2^e with S * sqrt(max y~^2) * sqrt(max|d| of the row) just below the FP16 maximum, so zh cannot overflow;
// zl stays a normal FP16 number for every entry within ~2^-11 of the bound (smaller ones lose low bits that do
// not matter at their size). The scale is per ROW (not per call) so that a row's arithmetic does not depend on
// which rows share its launch: row-sharded runs stay bitwise equal to single-GPU runs.
__device__ __forceinline__ int gram_scale_exp(float max_y2, float max_d) {
    const float m = sqrtf(max_y2) * sqrtf(max_d);
    if (!(m > 0.0f) || !(m < 3.0e38f)) return 0;
    int e = (int)floorf(log2f(60000.0f / m));
    return e > 40 ? 40 : (e < -40 ? -40 : e);  // S^2 and 1/S^2 stay finite
}

}  // namespace tc
}  // namespace wmf
