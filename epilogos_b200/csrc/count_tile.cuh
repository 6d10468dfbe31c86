// The count tile: 128 bins x 128 bytes in shared memory, row b = the 2K count bytes of bin b (uint16 little-endian pairs,
// zero padded), 16-byte chunks XOR-swizzled by (b mod 8) -- the SWIZZLE_128B operand layout of tcgen05.mma.  Read K-major
// it is a [128 bin] x [2K byte] A operand (S2 scores); read MN-major it is a [2K byte-index] x [128 bin] operand whose
// contraction index is the bin, i.e. both operands of the Gram update G += T T^t that yields the S2 expected table
// (expected.py:146-158).  Used by tc_tables.cu (K2 and K5).
#pragma once
#include "tc05.cuh"

namespace epi {

#ifdef __CUDACC__

constexpr int T2_OP_BYTES = 128 * 128;
constexpr int T2_DRAIN = 256;         // tiles between accumulator drains: 255*255*32768 < 2^31

// SM100 shared-memory descriptor of an MN-major SWIZZLE_128B operand whose MN extent is one 128-byte atom:
// 8 contraction rows of 128 bytes per 1024-byte atom (SBO), atoms stacked along the contraction index.
__device__ __forceinline__ uint64_t make_mnmajor_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)((128u >> 4) & 0x3fff) << 16;       // LBO: next 128-byte MN block (unused, one block)
    d |= (uint64_t)((1024u >> 4) & 0x3fff) << 32;      // SBO: next group of 8 contraction rows
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
constexpr uint32_t UMMA_A_MN_MAJOR = 1u << 15, UMMA_B_MN_MAJOR = 1u << 16;

// the count row of one bin (KT/2 words of uint16 pairs) -> its 128-byte operand row; `ones_word`/`ones_val` put the
// constant 1 of the N1 column into byte 2K (K2 only)
template <int KT>
__device__ __forceinline__ void store_operand_row(uint8_t* row_ptr, int r, const uint32_t (&cw)[KT / 2], int ones_word,
                                                  uint32_t ones_val) {
    constexpr int NW = ((KT / 2 + 1 + 3) / 4) * 4;     // words incl. the ones byte, whole 16-byte chunks
#pragma unroll
    for (int q = 0; q < NW / 4; ++q) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            w[i] = (4 * q + i < KT / 2) ? cw[4 * q + i] : 0u;
            if (4 * q + i == ones_word) w[i] |= ones_val;
        }
        *reinterpret_cast<uint4*>(row_ptr + ((q ^ (r & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// count row -> KT/2 words of uint16 pairs.  KR = compile-time state count (0: runtime K <= KT); an even KR makes the row a
// whole number of 4-byte words (LDS.32, no predicates).
template <int KT, int KR>
__device__ __forceinline__ void load_count_row(const uint16_t* row, int K, uint32_t (&cw)[KT / 2]) {
    if constexpr (KR != 0 && KR % 2 == 0) {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(row);
#pragma unroll
        for (int i = 0; i < KT / 2; ++i) cw[i] = i < KR / 2 ? w[i] : 0u;
    } else if constexpr (KR != 0) {
        // odd row length (15 states: 30-byte rows): the row starts on a 4-byte boundary only for even bins.  Read the
        // (KR + 1) / 2 aligned words that cover it and realign with funnel shifts: 8 LDS.32 + 8 SHF instead of 15 LDS.U16
        // + their merges (the halfword loads also bank-conflict at this pitch).
        constexpr int NW = (KR + 1) / 2;
        const uintptr_t a = reinterpret_cast<uintptr_t>(row);
        const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        const uint32_t sh = (a & 2) ? 16u : 0u;
        uint32_t t[NW];
#pragma unroll
        for (int i = 0; i < NW; ++i) t[i] = w[i];
#pragma unroll
        for (int i = 0; i < KT / 2; ++i) {
            if (i < NW - 1) cw[i] = __funnelshift_r(t[i], t[i + 1], sh);
            else if (i == NW - 1) cw[i] = (sh ? (t[i] >> 16) : t[i]) & 0xffffu;      // last state + nothing
            else cw[i] = 0u;
        }
    } else {
#pragma unroll
        for (int i = 0; i < KT / 2; ++i)
            cw[i] = (2 * i < K ? (uint32_t)row[2 * i] : 0u) | ((2 * i + 1 < K ? (uint32_t)row[2 * i + 1] : 0u) << 16);
    }
}
template <int KT>
__device__ __forceinline__ void load_count_row_guarded(const uint16_t* row, int K, bool live, uint32_t (&cw)[KT / 2]) {
#pragma unroll
    for (int i = 0; i < KT / 2; ++i)
        cw[i] = (live && 2 * i < K ? (uint32_t)row[2 * i] : 0u) | ((live && 2 * i + 1 < K ? (uint32_t)row[2 * i + 1] : 0u) << 16);
}

// Accumulator rows m = 2s (low-byte row of state s) and 2s+1 (high-byte row) live in adjacent lanes; lane 2s combines
// them into N2[s][.] and N1[s] (the ones column is column 2K) and adds them to the global int64 tables.  No smem.
template <int NCOL>
__device__ __forceinline__ void drain_gram(uint32_t tmem_lane_base, int warp, int lane, int K, unsigned long long* n1,
                                           unsigned long long* n2) {
    uint32_t v[NCOL];
#pragma unroll
    for (int c0 = 0; c0 < NCOL; c0 += 16) {
        uint32_t t16[16];
        tmem_ld_32x16(tmem_lane_base + (uint32_t)c0, t16);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[c0 + j] = t16[j];
    }
    const int m = warp * 32 + lane;
    const int s = m >> 1;
    const bool owner = (m & 1) == 0 && s < K;
    long long diag = 0, cnt1 = 0;
#pragma unroll
    for (int q = 0; q < NCOL / 2; ++q) {
        const uint32_t p0 = __shfl_down_sync(0xffffffffu, v[2 * q], 1), p1 = __shfl_down_sync(0xffffffffu, v[2 * q + 1], 1);
        const long long val = (long long)v[2 * q] + 256ll * (long long)v[2 * q + 1] + 256ll * ((long long)p0 + 256ll * (long long)p1);
        if (q == K) cnt1 = val;                                   // sum_b c_bs
        else if (q == s) diag = val;                              // sum_b c_bs^2
        else if (owner && q < K && n2 != nullptr && val != 0) atomicAdd(&n2[s * K + q], (unsigned long long)val);
    }
    if (owner) {
        diag -= cnt1;                                             // c*(c-1) on the diagonal
        if (n2 != nullptr && diag != 0) atomicAdd(&n2[s * K + s], (unsigned long long)diag);
        if (n1 != nullptr && cnt1 != 0) atomicAdd(&n1[s], (unsigned long long)cnt1);
    }
}


#endif  // __CUDACC__

}  // namespace epi
