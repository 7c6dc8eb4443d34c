// tc05.cuh -- tcgen05 / TMEM / UMMA shared-memory descriptor primitives (inline PTX) shared by the tensor-core kernels
// (gemm_tc.cu: kind::f16 GEMM with exact-integer f16 operands, fattn_tc.cu: flash attention, gemm_f16_tc.cu: F16/BF16 weight GEMM)
// and the 2-D / 3-D TMA tile loads the F16/BF16 weight kernels stream through (gemm_f16_tc.cu, gemv_f16.cu).
#pragma once
#include "common.cuh"

// ---- tcgen05 / TMEM primitives (inline PTX; SASS: UTCIMMA, LDTM, UTCBAR, ...) ------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// D[tmem] (+)= A[smem] * B[smem], int8 x int8 -> int32
__device__ __forceinline__ void mma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
    return d;                               // base offset 0, lbo mode 0, layout type 0 = no swizzle
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, "
        "%20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[smem] * B[smem], f16 x f16 -> f32 (SASS: UTCHMMA)
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 8 consecutive 32-bit columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], tf32 x tf32 -> f32, K = 8 per instruction (the low 13 mantissa bits of the operands are ignored)
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 16 consecutive 32-bit columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
                   "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
}

// K-major operand tile written by a SWIZZLE_128B TMA load: rows of 64 16-bit elements (128 bytes), 16-byte chunk c of row r stored at
// chunk c ^ (r & 7), 8-row groups 1024 bytes apart (SBO).  The tile base must be 1024-byte aligned; a K step of 16 elements inside the
// 128-byte row advances the start address by 32 bytes (the swizzle is applied to the computed address).
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;                 // LBO (unused for swizzled K-major layouts)
    d |= (uint64_t)(1024 >> 4) << 32;       // SBO: 8 rows x 128 bytes
    d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                 // layout type 2 = SWIZZLE_128B
    return d;
}
// instruction descriptor of tcgen05.mma kind::f16: f32 accumulator, K-major A and B, f16 (bf16 = false) or bf16 operands, M x N tile
__host__ __device__ constexpr uint32_t idesc_f16(bool bf16, int m, int n) {
    return (1u << 4) | (bf16 ? (1u << 7) | (1u << 10) : 0u) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// mbarrier wait that gives up after ~1 s (trap -> launch failure) instead of hanging the device on a pipeline bug
__device__ __forceinline__ void mbar_wait_bounded(uint64_t *bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 24)) __trap();
    }
}
// one lane of a fully converged warp (the single-thread roles keep their loops warp-uniform and predicate only the issue)
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}
// 2-D TMA tile load (SASS: UTMALDG): box at element coordinates (c0 = inner, c1 = outer) of the tensor map `tmap` (a __grid_constant__
// kernel parameter); out-of-bounds elements are written as zeros and still count toward the transaction bytes
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const void *tmap, int c0, int c1, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(smem_dst)),
                 "l"((uint64_t)(uintptr_t)tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
// 3-D TMA tile load: box at (c0 = inner, c1 = outer, c2 = depth), e.g. (k, row, expert) of a stack of expert matrices; with a box depth
// of 1 the shared-memory image is that of the 2-D box, and the zero fill stops at each matrix's own last row
__device__ __forceinline__ void tma_load_3d(void *smem_dst, const void *tmap, int c0, int c1, int c2, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(smem_u32(smem_dst)),
                 "l"((uint64_t)(uintptr_t)tmap), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
                 : "memory");
}
