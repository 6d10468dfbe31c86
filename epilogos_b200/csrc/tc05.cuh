// tcgen05 / TMEM wrappers shared by the tensor-core kernels (S3 Gram, S2 expected table, S2 scores).  sm_100a only.
#pragma once
#include "common.cuh"

namespace epi {

#ifdef __CUDACC__

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// generic-proxy writes to shared memory (st.shared) -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// bulk store shared -> global (16-byte aligned, size a multiple of 16), tracked by the thread's bulk async-group
__device__ __forceinline__ void bulk_store_1d(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reinterpret_cast<uint64_t>(gdst)),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// named barrier for a subset of the CTA's warps (id 1..15; nthreads a multiple of 32)
__device__ __forceinline__ void named_barrier(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// mbarrier wait: try_wait with a suspend-time hint so that a waiting warp sleeps in hardware instead of burning issue
// slots in a polling loop, plus a watchdog: a protocol bug traps (launch error) instead of hanging the GPU
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t hint_ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(hint_ns)
        : "memory");
    return ok != 0;
}
// suspend-time hint of mbar_wait_wd in ns (K5-S2 ran within 1 % at 0 / 500 / 5000 / 200000 ns, profiles/README.md)
constexpr uint32_t MBAR_WAIT_HINT_NS = 200000u;
__device__ __forceinline__ void mbar_wait_wd(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait_hint(bar, parity, MBAR_WAIT_HINT_NS)) {
        if (++spins > (1u << 22)) __trap();
    }
}
// latency-critical waits (the single MMA-issuing thread): plain polling, no suspend
__device__ __forceinline__ void mbar_wait_spin_wd(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 28)) __trap();
    }
}

// D[tmem] (+)= A[smem] * B[smem], int8 x int8 -> int32, issued by ONE thread
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}
// mbarrier arrives once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread i <- TMEM lane base+i)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    tmem_ld_wait();
}
// 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
    tmem_ld_wait();
}

// K-major operand tile in shared memory, 128-byte swizzle: rows of 128 bytes, 8-row atoms 1024 bytes apart.
// (SM100 UMMA shared-memory descriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48),
//  layout type SWIZZLE_128B = 2 [61,64).)  Byte (row, k) of the tile lives at
//      row*128 + (((k >> 4) ^ (row & 7)) << 4) + (k & 15)            (tile base 1024-byte aligned)
// which is what TMA's SWIZZLE_128B produces and what hand-written operand tiles must reproduce.
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)((1024u >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__host__ __device__ __forceinline__ uint32_t sw128_offset(uint32_t row, uint32_t k) {
    return row * 128u + ((((k >> 4) ^ (row & 7u)) << 4) | (k & 15u));
}

// instruction descriptor, kind::i8: D=S32 (2<<4), A=U8, B=U8 (format 0), both K-major, N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t umma_i8_idesc(uint32_t m, uint32_t n) {
    return (2u << 4) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

#endif  // __CUDACC__

}  // namespace epi
