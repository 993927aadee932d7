// Raw PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (MMA, TMEM).
// No CUTLASS dependency; bit layouts follow the PTX ISA "tcgen05" chapter.
#pragma once
#include <cstdint>
#include <cuda.h>

namespace evz {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes or the
// hint expires, instead of spinning through issue slots the epilogue warps need
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) { }
}
// spinning wait (test_wait never suspends the thread): for waits on the critical path of a kernel that has
// issue slots to spare -- waking up from a suspended try_wait costs far more than the poll loop
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity) {
    while (!mbar_test(bar, parity)) { __nanosleep(20); }      // short back-off: leave the issue slots to the warps that compute
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load: c0 = innermost coordinate (bytes for a u8 tensor), c1 = row
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
// L2 prefetch of a 2-D tile / of a linear range: no shared memory, no completion tracking
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* m, int c0, int c1) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
                 :: "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_1d(const void* gsrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes) : "memory");
}
// 1-D bulk copy global -> shared (16-byte aligned, size multiple of 16)
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_u32(smem_result)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major operand tile in shared memory, 128-byte rows, SWIZZLE_128B (as written by a TMA
// box of 128 bytes x R rows with CU_TENSOR_MAP_SWIZZLE_128B): 8-row x 128-byte atoms,
// stride between atoms along M/N (SBO) = 1024 bytes, one atom along K (LBO unused).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr_bytes & 0x3FFFF) >> 4);        // start address   [0,14)
    d |= static_cast<uint64_t>(0) << 16;                                 // LBO             [16,30)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;                         // SBO             [32,46)
    d |= static_cast<uint64_t>(1) << 46;                                 // version = 1 (sm_100)
    d |= static_cast<uint64_t>(2) << 61;                                 // layout = SWIZZLE_128B
    return d;
}
// Instruction descriptor for kind::i8: u8 x u8 -> s32, both operands K-major.
__host__ __device__ constexpr uint32_t umma_idesc_u8(uint32_t m, uint32_t n) {
    return (2u << 4)            // c_format  = S32
         | (0u << 7)            // a_format  = unsigned 8-bit
         | (0u << 10)           // b_format  = unsigned 8-bit
         | (0u << 15) | (0u << 16)   // K-major A, B
         | ((n >> 3) << 17)     // n_dim
         | ((m >> 4) << 24);    // m_dim
}
// D[tmem] (+)= A[smem] . B[smem]^T, one 128 x N x 32 step; issued by ONE thread.
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 :: "r"(smem_u32(bar)) : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive 32-bit columns.
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
}
// wait for outstanding tcgen05.ld and make the destination registers depend on the wait, so that
// neither nvcc nor ptxas can schedule a use of them ahead of it
__device__ __forceinline__ void tmem_ld_wait_dep(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31]));
}

__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}

}  // namespace evz
