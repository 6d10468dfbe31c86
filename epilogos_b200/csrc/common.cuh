// Shared helpers for the epilogos_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/epilogos_b200.h"

namespace epi {

// ---- error plumbing ---------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_device();   // 0 if an sm_100 device is current, else sets the error and returns non-zero

#define EPI_CUDA(call)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            epi::set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,               \
                           cudaGetErrorString(e__));                                          \
            return 1;                                                                         \
        }                                                                                     \
    } while (0)

#define EPI_REQUIRE(cond, ...)                                                                \
    do {                                                                                      \
        if (!(cond)) {                                                                        \
            epi::set_error(__VA_ARGS__);                                                      \
            return 2;                                                                         \
        }                                                                                     \
    } while (0)

int sm_count();
unsigned grid_for(long long n, int per_block, int per_sm);   // min(ceil(n / per_block), SMs * per_sm), at least 1
int persistent_grid(int64_t ntiles, int per_sm);   // min(ntiles, SMs * per_sm), at least 1

// ---- per-device workspace ---------------------------------------------------------------------
constexpr int S1_TABLE_MAX_WIDTH = 4095;           // widest input whose S1 scores come from a value table

struct PrepFlags {
    int has_zero;       // some expected frequency is 0 -> masked terms -> DIRECT evaluation
};

// constants of the kind::i8 S2 score kernel (tc_tables.cu), written by its prepare kernel
struct K5TcConsts {
    double dg[EPI_MAX_STATES];                  // M_tt 2^-F / perms / 8: the [s==t] term of y_t (see `base` in the kernel)
    double scale;                               // 2^-F / perms
    double cst;                                 // (2^52 + 2^51) * scale
    int has_zero;
    uint32_t m1, m8, m16;                       // 1, 2^8, 2^16 (opaque to the compiler)
    int fbits;                                  // F: M = round(-log2 E * 2^F)
};

// Small tables the score and normalise entry points stage on the device before a launch.  One per device, allocated on
// first use; calls for one device are stream-ordered with respect to each other (include/epilogos_b200.h).
struct DeviceWorkspace {
    unsigned long long reduce_slots[64];                            // grand totals of epi_normalize_i64, round-robin
    double log2e[EPI_MAX_STATES * EPI_MAX_STATES];                  // K5: log2 E, copied to constant memory
    PrepFlags prep_flags;                                           // K5: zero flag of the expected table
    int s3_symmetric;                                               // K6: the S3 terms table is symmetric
    alignas(16) uint8_t k5tc_b_image[8 * EPI_MAX_STATES * 128];     // kind::i8 B operand: 8 rows x 128 B per state
    K5TcConsts k5tc_consts;
    alignas(8) double s1_v64[EPI_MAX_STATES * (S1_TABLE_MAX_WIDTH + 1)];   // S1 value table [K][width + 1]
    alignas(8) float s1_v32[EPI_MAX_STATES * (S1_TABLE_MAX_WIDTH + 1)];    // its float32 rounding
    alignas(8) float perm_v32[2][EPI_MAX_STATES * (S1_TABLE_MAX_WIDTH + 1)];  // permutations.cu: the tables of A', B'
};
static_assert(offsetof(DeviceWorkspace, k5tc_b_image) % 16 == 0, "the B operand image is a bulk-copy source");
static_assert(offsetof(DeviceWorkspace, s1_v64) % 8 == 0 && offsetof(DeviceWorkspace, s1_v32) % 8 == 0,
              "the S1 value tables need 8-byte alignment");

DeviceWorkspace* device_workspace();   // the current device's workspace; nullptr if it could not be allocated

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda dependency)
typedef CUresult (*tensor_map_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                         const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                         CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                         CUtensorMapFloatOOBfill);
tensor_map_encode_fn get_tensor_map_encode();

// K5-S1 value table [K][width + 1] of the expected table e (scores.cu): the float64 reference expression and its float32
// rounding, the values epi_scores_s1 looks up in TABLE mode; width <= S1_TABLE_MAX_WIDTH
int s1_value_table(const float* e, int K, int width, float* v32, double* v64, cudaStream_t st);

// tensor-core forms of the S2 table contractions (tc_tables.cu)
int launch_k2_tc(const uint16_t* cnt, int64_t bins, int K, int64_t* n1, int64_t* n2, cudaStream_t st);
int scores_s2_tc(const uint16_t* cnt, int64_t bins, int K, int width, int64_t perms, const float* e, int* zero_flag,
                 float* o32, double* o64, cudaStream_t st);
bool scores_s2_tc_eligible(int width);
int scores_s2_tc_fixed_point(const float* e, int K, int64_t perms, unsigned long long* mfix_dev, int* fbits_host,
                             cudaStream_t st);

// ---- device-side PTX wrappers -----------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Release of a shared-memory buffer to an asynchronous producer (TMA / bulk copy): the arrive must not be performed before
// the loads that read the buffer have returned.  An arrive issued right behind the loads can overtake them (measured in
// tc_tables.cu: corrupted rows), so these variants take a value that DEPENDS on the loaded data as an (unused) operand:
// the instruction cannot issue until that value exists, i.e. until the loads have completed.
__device__ __forceinline__ void mbar_arrive_after(uint64_t* bar, uint32_t dep) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)), "r"(dep) : "memory");
}
__device__ __forceinline__ void mbar_arrive_after(uint64_t* bar, double dep) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)), "d"(dep) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// 2D tiled TMA load global -> shared, completion signalled on an mbarrier (cp.async.bulk.tensor)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int32_t c0, int32_t c1,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// 1D bulk copy global -> shared (16-byte aligned source, destination and size), completion on an mbarrier
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ uint32_t lop3_xor3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t lop3_maj(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xe8;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

// Philox4x32-10 counter-based generator (paired null shuffles, pairwise.cu; null subsampling, pairwise_stats.cu)
struct Philox {
    uint32_t key0, key1;
    uint32_t ctr[4];
    uint32_t out[4];
    int have;

    __device__ __forceinline__ void round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) const {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    }
    __device__ __forceinline__ void refill() {
        uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
        uint32_t k0 = key0, k1 = key1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            round(c, k0, k1);
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
        ++ctr[0];
        have = 4;
    }
    __device__ __forceinline__ uint32_t next() {
        if (have == 0) refill();
        return out[--have];
    }
};

#endif  // __CUDACC__

}  // namespace epi
