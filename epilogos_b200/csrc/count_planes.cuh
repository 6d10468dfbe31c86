// Bit-sliced label counting shared by K1 (counts.cu) and the column-group counts (groups.cu): one-hot words of the labels
// are summed with a carry-save adder tree into counter planes, the planes are flushed into packed 16-bit counters, and the
// counters are unpacked into per-state counts.  A "source" supplies the words: Src::tword<I>() is the I-th summed word.
//   MODE_F2   <= 16 states: two-bit fields, three one-hot words summed per word (field values <= 3)
//   MODE_F2M  17 or 18 states: as F2; states 16 / 17 alias fields 0 / 1 and are separated with sum(v) and sum(v^2)
//   MODE_B1   19..32 states: one-bit fields, one one-hot word per label
#pragma once
#include "common.cuh"

namespace epi {

#ifdef __CUDACC__

enum { MODE_F2 = 0, MODE_F2M = 1, MODE_B1 = 2 };

template <int MODE>
struct PlaneCount {
    static constexpr int N = (MODE == MODE_B1) ? 10 : 9;        // bit-sliced counter depth
    static constexpr int CAP = (1 << N) - 1;                    // words that may be added before a flush
};

// Depth-first carry-save tree: Tree<L>::get<I> folds 2^L consecutive words into planes p[0..L-1] and
// returns the carry word of weight 2^L.
template <int L>
struct Tree {
    template <int I, class Src, int NP>
    static __device__ __forceinline__ uint32_t get(const Src& src, uint32_t (&p)[NP]) {
        uint32_t a = Tree<L - 1>::template get<2 * I>(src, p);
        uint32_t b = Tree<L - 1>::template get<2 * I + 1>(src, p);
        uint32_t s = lop3_xor3(p[L - 1], a, b);
        uint32_t c = lop3_maj(p[L - 1], a, b);
        p[L - 1] = s;
        return c;
    }
};
template <>
struct Tree<0> {
    template <int I, class Src, int NP>
    static __device__ __forceinline__ uint32_t get(const Src& src, uint32_t (&)[NP]) {
        return src.template tword<I>();
    }
};

// Fold N words of weight 2^L into planes p[L..]; odd leftovers go through a half adder.
template <int L, int N, int NP>
struct Reduce {
    static __device__ __forceinline__ void run(const uint32_t (&w)[N], uint32_t (&p)[NP]) {
        if constexpr (L >= NP - 1) {
#pragma unroll
            for (int i = 0; i < N; ++i) p[NP - 1] ^= w[i];
        } else {
            constexpr int NPAIR = N / 2;
            constexpr int NN = NPAIR + (N & 1);
            uint32_t nx[NN];
#pragma unroll
            for (int i = 0; i < NPAIR; ++i) {
                uint32_t s = lop3_xor3(p[L], w[2 * i], w[2 * i + 1]);
                nx[i] = lop3_maj(p[L], w[2 * i], w[2 * i + 1]);
                p[L] = s;
            }
            if constexpr (N & 1) {
                nx[NPAIR] = p[L] & w[N - 1];
                p[L] ^= w[N - 1];
            }
            Reduce<L + 1, NN, NP>::run(nx, p);
        }
    }
};

// bit-sliced planes -> packed 16-bit counters, then clear the planes
template <int MODE, int NP, int NACC>
__device__ __forceinline__ void flush_planes(uint32_t (&p)[NP], uint32_t (&acc)[NACC]) {
#pragma unroll
    for (int k = 0; k < NP; ++k) {
#pragma unroll
        for (int f = 0; f < NACC; ++f) {
            // lo half: state/field f, hi half: state f+16 / field f+8.  acc += t * 2^k as one IMAD.
            const uint32_t t = (MODE == MODE_B1) ? ((p[k] >> f) & 0x00010001u) : ((p[k] >> (2 * f)) & 0x00030003u);
            asm("mad.lo.u32 %0, %1, %2, %0;" : "+r"(acc[f]) : "r"(t), "r"(1u << k));
        }
        p[k] = 0;
    }
}

// Zeroed counters, except that the low half of acc[0] starts at 0x10000 - npad: the npad zero labels that are counted but
// are not data (the padding of a row or of a column list to whole chunks) carry it exactly once into the high half, so the
// low half ends at the data's own count of field 0 however close the padded row comes to 65,535 labels or goes past it.
// unpack_counts takes that one carry back out.
template <int NACC>
__device__ __forceinline__ void init_counters(uint32_t (&acc)[NACC], int npad) {
    acc[0] = 0x10000u - (uint32_t)npad;
#pragma unroll
    for (int f = 1; f < NACC; ++f) acc[f] = 0;
}

// packed counters (started by init_counters) -> per-state counts cs[0..EPI_MAX_STATES).  sum1 / sum2 (MODE_F2M only) are
// sum(v) and sum(v^2) over the counted labels.
template <int MODE, int NACC>
__device__ __forceinline__ void unpack_counts(const uint32_t (&acc)[NACC], uint32_t sum1, uint32_t sum2,
                                              uint32_t (&cs)[EPI_MAX_STATES]) {
    // the pad's carry leaves acc[0] modulo 2^32: a high-half count of 65,535 had wrapped to 0 and comes back
    const auto word = [&](int f) { return f == 0 ? acc[0] - 0x10000u : acc[f]; };
    if constexpr (MODE == MODE_B1) {
#pragma unroll
        for (int f = 0; f < 16; ++f) {
            cs[f] = word(f) & 0xffffu;
            cs[f + 16] = word(f) >> 16;
        }
    } else {
#pragma unroll
        for (int f = 0; f < 8; ++f) {
            cs[f] = word(f) & 0xffffu;
            cs[f + 8] = word(f) >> 16;
        }
#pragma unroll
        for (int f = 16; f < EPI_MAX_STATES; ++f) cs[f] = 0;
        if constexpr (MODE == MODE_F2M) {
            // states 16 and 17 landed in fields 0 and 1; separate them with sum(v) and sum(v^2)
            uint32_t m1 = 0, m2 = 0;
#pragma unroll
            for (int f = 1; f < 16; ++f) {
                m1 += f * cs[f];
                m2 += f * f * cs[f];
            }
            const uint32_t hi = (sum1 - m1) >> 4;                    // c16 + c17
            const uint32_t c17 = ((sum2 - m2) - 256u * hi) >> 5;     // 256*c16 + 288*c17 - 256*(c16+c17)
            const uint32_t c16 = hi - c17;
            cs[16] = c16;
            cs[17] = c17;
            cs[0] -= c16;
            cs[1] -= c17;
        }
    }
}

#endif  // __CUDACC__

}  // namespace epi
