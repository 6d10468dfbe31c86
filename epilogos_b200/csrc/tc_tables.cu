// Tensor-core forms of the two count-table contractions of the S2 path (tcgen05.mma kind::i8, exact int32
// accumulation in TMEM).  A uint16 count is two unsigned bytes, so the per-bin count row IS an int8 operand:
//
//   K2 (expected.py:146-158, s2Calc)     N2[s][t] = sum_b c_bs c_bt - [s==t] c_bs
//        G = Bt B over the bins, B[b][2s+h] = byte h of c_bs  ->  N2[s][t] = sum_{h,h'} 256^(h+h') G[2s+h][2t+h'];
//        a row of ones appended to the operand gives N1[s] = sum_b c_bs in the same pass.
//   K5 (scores.py:412, 443-451, s2Score) the 18x18 mat-vec  y_t = sum_s c_s (-log2 E_st)  of the TABLE evaluation
//        (csrc/scores.cu) with -log2 E in 56-bit fixed point split into seven base-256 digits:
//        D[b][8t+d] = sum_s lo(c_bs) dig_d(M_st) + hi(c_bs) dig_{d-1}(M_st),   Y_bt = sum_d 256^d D[b][8t+d]
//        is the exact integer sum_s c_bs M_st; the float64 epilogue adds the O(K) remainder of the score formula.
//
// Both replace ALU / fp64-pipe loops that were the limiters of K2 (IMAD) and K5 (324 DFMA per bin); what is left per
// bin is byte shuffling for K2 and ~7 fp64 operations per state for K5.
#include "common.cuh"
#include "tc05.cuh"
#include "count_tile.cuh"

namespace epi {

// ================================================================================================
// K2 on the tensor cores
//
// Operand tile = 128 bins x 128 bytes: row b holds the 2K count bytes of bin b (zero padded), 16-byte chunks XOR-swizzled
// by (b mod 8).  Read as an MN-major SWIZZLE_128B operand this is a [128 byte-index] x [128 bin] matrix with the bin
// as the contraction index, so the tile is BOTH operands of G += T T^t and needs no transposition; the very same tile
// read K-major is the A operand of the score kernel below.  Byte column 2K of every row is 1 (the N1 column).
// ================================================================================================
constexpr int T2_BINS = 128;          // bins per tile
constexpr int T2_STAGES = 4;          // count-tile ring (1D bulk copies)
constexpr int T2_OPS = 2;             // operand buffers
constexpr int T2_THREADS = 192;       // warps 0-3 build operand rows, warp 4 = copy producer, warp 5 = MMA issuer
constexpr int T2_TMEM_COLS = 128;

template <int KT, int KR>
__global__ void __launch_bounds__(T2_THREADS, 4)
k2_tc_kernel(const uint16_t* __restrict__ cnt, long long bins, int Krt, unsigned long long* __restrict__ n1,
             unsigned long long* __restrict__ n2) {
    const int K = KR ? KR : Krt;
    constexpr int NCOL = ((2 * KT + 1) + 15) & ~15;                 // UMMA N: count bytes + the ones column
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int tile_bytes = T2_BINS * K * 2;                         // multiple of 256
    uint8_t* ops = smem;                                            // T2_OPS x [128 bins x 128 B]
    uint8_t* ring = ops + T2_OPS * T2_OP_BYTES;
    uint64_t* ld_full = reinterpret_cast<uint64_t*>(ring + T2_STAGES * tile_bytes);
    uint64_t* ld_empty = ld_full + T2_STAGES;
    uint64_t* op_full = ld_empty + T2_STAGES;
    uint64_t* op_empty = op_full + T2_OPS;
    uint64_t* acc_full = op_empty + T2_OPS;
    uint64_t* acc_empty = acc_full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long ntiles = (bins + T2_BINS - 1) / T2_BINS;
    const long long nfull = bins / T2_BINS;

    for (int i = tid; i < T2_OPS * T2_OP_BYTES / 16; i += T2_THREADS)
        reinterpret_cast<uint4*>(ops)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();
    if (tid == 0) {
        for (int s = 0; s < T2_STAGES; ++s) {
            mbar_init(&ld_full[s], 1);
            mbar_init(&ld_empty[s], 4);
        }
        for (int o = 0; o < T2_OPS; ++o) {
            mbar_init(&op_full[o], 4);
            mbar_init(&op_empty[o], 1);
        }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, 2);
        mbar_fence_init();
    }
    if (warp == 5) tmem_alloc(tmem_slot, T2_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 4) {
        // ------------------------------ bulk-copy producer ------------------------------
        if (lane == 0) {
            int i = 0;
            for (long long t = blockIdx.x; t < nfull; t += gridDim.x, ++i) {
                const int s = i % T2_STAGES;
                mbar_wait_wd(&ld_empty[s], (((uint32_t)(i / T2_STAGES)) & 1u) ^ 1u);
                mbar_expect_tx(&ld_full[s], (uint32_t)tile_bytes);
                bulk_load_1d(ring + s * tile_bytes, cnt + t * (long long)T2_BINS * K, (uint32_t)tile_bytes, &ld_full[s]);
            }
        }
    } else if (warp == 5) {
        // ------------------------------ MMA issuer (one thread) ------------------------------
        if (lane == 0) {
            const uint32_t idesc = umma_i8_idesc(128, NCOL) | UMMA_A_MN_MAJOR | UMMA_B_MN_MAJOR;
            uint32_t acc = 0, dph = 0;
            int i = 0;
            for (long long t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
                const int o = i % T2_OPS;
                mbar_wait_spin_wd(&op_full[o], ((uint32_t)(i / T2_OPS)) & 1u);
                tc_fence_after();
                const uint64_t desc = make_mnmajor_sw128_desc(smem_u32(ops + o * T2_OP_BYTES));
#pragma unroll
                for (int k = 0; k < T2_BINS / 32; ++k) {
                    // 32 bins = 4 atoms of 1024 bytes further along the contraction index
                    umma_i8(tmem_base, desc + 256 * k, desc + 256 * k, idesc, acc);      // A and B are the same tile
                    acc = 1;
                }
                umma_commit(&op_empty[o]);
                if ((i + 1) % T2_DRAIN == 0 || t + gridDim.x >= ntiles) {
                    umma_commit(acc_full);
                    mbar_wait_spin_wd(acc_empty, dph);
                    dph ^= 1;
                    tc_fence_after();
                    acc = 0;
                }
            }
        }
    } else {
        // ------------------------------ operand builders: one bin per thread ------------------------------
        uint32_t dph = 0;
        int i = 0;
        for (long long t = blockIdx.x; t < ntiles; t += gridDim.x, ++i) {
            const int s = i % T2_STAGES, o = i % T2_OPS;
            uint32_t cw[KT / 2];
            if (t < nfull) {
                mbar_wait_wd(&ld_full[s], ((uint32_t)(i / T2_STAGES)) & 1u);
                load_count_row<KT, KR>(reinterpret_cast<const uint16_t*>(ring + s * tile_bytes) + tid * K, K, cw);
            } else {
                const long long b = t * T2_BINS + tid;
                load_count_row_guarded<KT>(cnt + b * K, K, b < bins, cw);
            }
            mbar_wait_wd(&op_empty[o], (((uint32_t)(i / T2_OPS)) & 1u) ^ 1u);
            // byte 2K of the row = 1 for live bins (N1 column)
            const bool live = t * T2_BINS + tid < bins;
            store_operand_row<KT>(ops + o * T2_OP_BYTES + tid * 128, tid, cw, K / 2,
                                  live ? (1u << (16 * (K & 1))) : 0u);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&op_full[o]);
                if (t < nfull) mbar_arrive(&ld_empty[s]);      // released only after the loaded counts were consumed (see K5)
            }

            if ((i + 1) % T2_DRAIN == 0 || t + gridDim.x >= ntiles) {
                mbar_wait_wd(acc_full, dph);
                dph ^= 1;
                tc_fence_after();
                if (warp < 2) {
                    drain_gram<NCOL>(tmem_base + ((uint32_t)(warp * 32) << 16), warp, lane, K, n1, n2);
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_empty);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) tmem_dealloc(tmem_base, T2_TMEM_COLS);
}

template <int KT, int KR>
static int launch_k2_tc_impl(const uint16_t* cnt, int64_t bins, int K, int64_t* n1, int64_t* n2, cudaStream_t st) {
    const size_t smem = 1024 + (size_t)T2_OPS * T2_OP_BYTES + (size_t)T2_STAGES * T2_BINS * K * 2 +
                        (2 * T2_STAGES + 2 * T2_OPS + 2) * 8 + 16;
    auto kern = k2_tc_kernel<KT, KR>;
    EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t ntiles = (bins + T2_BINS - 1) / T2_BINS;
    const int ctas = 4;    // measured at 15.5 M bins x 18 states: 0.33 / 0.22 / 0.19 ms at 1 / 2 / 3 CTAs per SM (6 stages), 0.185 at 4 (4 stages)
    kern<<<persistent_grid(ntiles, ctas), T2_THREADS, smem, st>>>(cnt, (long long)bins, K,
                                                                reinterpret_cast<unsigned long long*>(n1),
                                                                reinterpret_cast<unsigned long long*>(n2));
    EPI_CUDA(cudaGetLastError());
    return 0;
}

int launch_k2_tc(const uint16_t* cnt, int64_t bins, int K, int64_t* n1, int64_t* n2, cudaStream_t st) {
    if (K == 18) return launch_k2_tc_impl<18, 18>(cnt, bins, K, n1, n2, st);
    if (K == 15) return launch_k2_tc_impl<16, 15>(cnt, bins, K, n1, n2, st);
    if (K <= 16) return launch_k2_tc_impl<16, 0>(cnt, bins, K, n1, n2, st);
    if (K <= 18) return launch_k2_tc_impl<18, 0>(cnt, bins, K, n1, n2, st);
    return launch_k2_tc_impl<32, 0>(cnt, bins, K, n1, n2, st);
}

// ================================================================================================
// K5 (S2) on the tensor cores
// ================================================================================================
constexpr int T5_BINS = 128;
constexpr int T5_A_BYTES = 128 * 128;
constexpr unsigned long long T5_MAGIC = 0x4338000000000000ull;      // bits of 2^52 + 2^51: integer <-> double without I2F
constexpr int T5_MAX_WIDTH = 2047;

__device__ __forceinline__ unsigned long long mad_wide(uint32_t a, uint32_t b, unsigned long long c) {
    unsigned long long d;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(d) : "r"(a), "r"(b), "l"(c));
    return d;
}

__device__ __forceinline__ uint32_t mad_lo(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__constant__ K5TcConsts c_k5tc;

// one CTA: float32 expected table -> fixed-point digits of -log2 E laid out as the 128-byte-swizzled B operand
// (row n = 8t + d, byte k = 2s + h holds digit d-h of M_st), per-state constants, zero flag; mfix_out (optional)
// receives the fixed-point table itself (diagnostic / tests).
__global__ void k5tc_prepare_kernel(const float* __restrict__ e, int K, double perms, int nrows,
                                    uint8_t* __restrict__ b_image, K5TcConsts* __restrict__ out, int* __restrict__ zero_flag,
                                    unsigned long long* __restrict__ mfix_out) {
    __shared__ unsigned long long mfix[EPI_MAX_STATES * EPI_MAX_STATES];
    __shared__ double mval[EPI_MAX_STATES * EPI_MAX_STATES];
    __shared__ unsigned long long maxbits;
    __shared__ int zero, fbits;
    if (threadIdx.x == 0) {
        maxbits = 0ull;
        zero = 0;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K * K; i += blockDim.x) {
        const double ev = (double)e[i];
        double m = 0.0;
        if (ev > 0.0) m = -log2(ev);
        else zero = 1;
        if (m < 0.0) m = 0.0;                      // E <= 1 always; guards -0.0
        mval[i] = m;
        atomicMax(&maxbits, (unsigned long long)__double_as_longlong(m));      // non-negative doubles order like integers
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double mx = __longlong_as_double((long long)maxbits);
        int ib = 1;
        while (ib < 12 && (double)(1ull << ib) <= mx) ++ib;       // mx < 2^ib
        fbits = 56 - ib;
    }
    __syncthreads();
    const int F = fbits;
    for (int i = threadIdx.x; i < K * K; i += blockDim.x) {
        unsigned long long v = (unsigned long long)llrint(ldexp(mval[i], F));
        if (v >= (1ull << 56)) v = (1ull << 56) - 1;
        mfix[i] = v;
        if (mfix_out != nullptr) mfix_out[i] = v;
    }
    for (int i = threadIdx.x; i < nrows * 128 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(b_image)[i] = 0u;
    __syncthreads();
    for (int i = threadIdx.x; i < K * K * 14; i += blockDim.x) {
        const int dd = i % 7, h = (i / 7) & 1, st = i / 14;
        const int s = st / K, t = st - s * K;
        const uint32_t n = (uint32_t)(t * 8 + dd + h), k = (uint32_t)(2 * s + h);
        b_image[sw128_offset(n, k)] = (uint8_t)((mfix[st] >> (8 * dd)) & 255ull);
    }
    if (threadIdx.x < K) out->dg[threadIdx.x] = ldexp((double)mfix[threadIdx.x * K + threadIdx.x], -F - 3) / perms;
    if (threadIdx.x == 0) {
        const double scale = ldexp(1.0, -F) / perms;
        out->scale = scale;
        out->cst = 6755399441055744.0 * scale;          // 2^52 + 2^51
        out->has_zero = zero;
        out->m1 = 1u;
        out->m8 = 1u << 8;
        out->m16 = 1u << 16;
        out->fbits = F;
        *zero_flag = zero;
    }
}

// KT: even unroll bound on the state index; KR: the state count when known at compile time (0 = runtime K <= KT);
// NWG: warpgroups = accumulator regions in TMEM; WANT64: also write the unrounded float64 scores (tests).
template <int KT, int KR, int NWG, bool WANT64>
__global__ void __launch_bounds__(NWG * 128 + 64, 1)
k5_s2_tc_kernel(const uint16_t* __restrict__ cnt, long long bins, int Krt, int width, double perms,
                const uint8_t* __restrict__ b_image, float* __restrict__ out32, double* __restrict__ out64) {
    if (c_k5tc.has_zero) return;          // masked terms: the DIRECT kernel launched behind this one does the work

    static_assert(KT % 2 == 0, "KT must be even");
    constexpr int NPAD = ((8 * KT + 31) / 32) * 32;          // TMEM columns per warpgroup
    static_assert(NPAD * NWG <= 512, "accumulator regions exceed TMEM");
    constexpr int KSTEPS = (2 * KT + 31) / 32;               // UMMA K steps (32 bytes each)
    const int K = KR ? KR : Krt;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int slab_bytes = T5_BINS * K * 2;                                  // multiple of 256
    uint8_t* a_ops = smem;                                                   // NWG x 16 KB
    uint8_t* b_op = a_ops + NWG * T5_A_BYTES;                                // NPAD x 128 B
    uint8_t* slabs = b_op + NPAD * 128;                                      // NWG x 2 x slab_bytes
    float* stage = reinterpret_cast<float*>(slabs + NWG * 2 * slab_bytes);   // NWG x 128 x K
    double* g1 = reinterpret_cast<double*>(stage + NWG * T5_BINS * K);       // width + 1 entries c HG[c] (+1 pad)
    double* f1 = g1 + ((width + 2) & ~1);                                    // width + 1 entries F[c] (+1 pad)
    uint64_t* ld_full = reinterpret_cast<uint64_t*>(f1 + ((width + 2) & ~1)); // [NWG][2]
    uint64_t* ld_empty = ld_full + NWG * 2;
    uint64_t* a_full = ld_empty + NWG * 2;                                   // [NWG]
    uint64_t* mma_done = a_full + NWG;                                       // [NWG]
    uint64_t* b_full = mma_done + NWG;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_full + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int NT = NWG * 128 + 64;
    const long long ntiles = (bins + T5_BINS - 1) / T5_BINS;
    const long long nfull = bins / T5_BINS;

    for (int i = tid; i < NWG * T5_A_BYTES / 16; i += NT) reinterpret_cast<uint4*>(a_ops)[i] = make_uint4(0u, 0u, 0u, 0u);
    {
        // F[c] = c log2(c) / P,  HG[c] = ((log2 c - log2 P)(W - 1) - c log2 c + (c-1) log2(c-1)) / P      (scores.cu header)
        // score_t = c_t (base_t + HG[c_t]) = fma(c_t, base_t, c_t HG[c_t]): the second table holds c HG[c]
        const double lp = log2(perms), invp = 1.0 / perms, wm1 = (double)width - 1.0;
        for (int c = tid; c <= width; c += NT) {
            const double l = c > 0 ? log2((double)c) : 0.0;
            const double l1 = c > 1 ? log2((double)(c - 1)) : 0.0;
            const double cl = (double)c * l;
            f1[c] = cl * invp;
            g1[c] = (double)c * ((fma(l - lp, wm1, -cl) + (double)(c > 0 ? c - 1 : 0) * l1) * invp);
        }
    }
    fence_proxy_async_smem();
    if (tid == 0) {
        for (int i = 0; i < NWG * 2; ++i) {
            mbar_init(&ld_full[i], 1);
            mbar_init(&ld_empty[i], 4);
        }
        for (int g = 0; g < NWG; ++g) {
            mbar_init(&a_full[g], 4);
            mbar_init(&mma_done[g], 1);
        }
        mbar_init(b_full, 1);
        mbar_fence_init();
    }
    if (warp == 4 * NWG + 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 4 * NWG) {
        // ------------------------------ bulk-copy producer ------------------------------
        if (lane == 0) {
            mbar_expect_tx(b_full, NPAD * 128);
            bulk_load_1d(b_op, b_image, NPAD * 128, b_full);
            int j = 0;
            for (long long t = blockIdx.x; t < nfull; t += gridDim.x, ++j) {
                const int g = j % NWG, u = j / NWG, b = u & 1;
                mbar_wait_wd(&ld_empty[g * 2 + b], (((uint32_t)(u >> 1)) & 1u) ^ 1u);
                mbar_expect_tx(&ld_full[g * 2 + b], (uint32_t)slab_bytes);
                bulk_load_1d(slabs + (g * 2 + b) * slab_bytes, cnt + t * (long long)T5_BINS * K, (uint32_t)slab_bytes,
                             &ld_full[g * 2 + b]);
            }
        }
    } else if (warp == 4 * NWG + 1) {
        // ------------------------------ MMA issuer (one thread) ------------------------------
        if (lane == 0) {
            const uint32_t nmma = (uint32_t)((8 * K + 15) & ~15);
            const uint32_t idesc = umma_i8_idesc(128, nmma);
            mbar_wait_wd(b_full, 0);
            const uint64_t b_desc = make_kmajor_sw128_desc(smem_u32(b_op));
            int j = 0;
            for (long long t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
                const int g = j % NWG, u = j / NWG;
                mbar_wait_spin_wd(&a_full[g], ((uint32_t)u) & 1u);
                tc_fence_after();
                const uint64_t a_desc = make_kmajor_sw128_desc(smem_u32(a_ops + g * T5_A_BYTES));
#pragma unroll
                for (int k = 0; k < KSTEPS; ++k)
                    umma_i8(tmem_base + (uint32_t)(g * NPAD), a_desc + 2 * k, b_desc + 2 * k, idesc, k ? 1u : 0u);
                umma_commit(&mma_done[g]);
            }
        }
    } else {
        // ------------------------------ warpgroups: one bin per thread ------------------------------
        const int g = warp >> 2, r = tid & 127;
        uint8_t* a_row = a_ops + g * T5_A_BYTES + r * 128;
        float* mystage = stage + g * T5_BINS * K;
        const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(g * NPAD);
        // everything that multiplies the count is kept divided by 8: the count enters as the double 8 c (its table byte offset)
        const double scale = c_k5tc.scale * 0.125, cst = c_k5tc.cst, scale32 = c_k5tc.scale * (4294967296.0 * 0.125);
        int u = 0;
        for (long long t = blockIdx.x + (long long)g * gridDim.x; t < ntiles; t += (long long)NWG * gridDim.x, ++u) {
            const long long bin0 = t * T5_BINS;
            const int b = u & 1;
            uint32_t cw[KT / 2];                       // the count row as uint16 pairs (state 2i in the low half)
            if (t < nfull) {
                mbar_wait_wd(&ld_full[g * 2 + b], ((uint32_t)(u >> 1)) & 1u);
                load_count_row<KT, KR>(reinterpret_cast<const uint16_t*>(slabs + (g * 2 + b) * slab_bytes) + r * K, K, cw);
            } else {
                load_count_row_guarded<KT>(cnt + (bin0 + r) * K, K, bin0 + r < bins, cw);
            }
            store_operand_row<KT>(a_row, r, cw, -1, 0u);        // the count row's bytes ARE the K-major A operand row
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&a_full[g]);
                // The slab is released only here, after the operand stores have CONSUMED every loaded count: an arrive
                // issued right behind the loads can be performed before they return (measured: corrupted rows when the
                // 30-byte row pitch of 15-state models makes the loads replay), and the producer would overwrite the slab.
                if (t < nfull) mbar_arrive(&ld_empty[g * 2 + b]);
            }

            // work that does not need the accumulators: A = sum_s F[c_s]      (c = 0 for s >= K: F[0] = 0)
            // byte offsets c_s * 8 into the two look-up tables, extracted once (both tables are indexed by the same counts)
            uint32_t co[KT];
#pragma unroll
            for (int s = 0; s < KT; ++s) co[s] = ((cw[s >> 1] >> (16 * (s & 1))) & 0xffffu) << 3;
            double a4[4] = {0.0, 0.0, 0.0, 0.0};       // four partial sums: the adds are ~20-cycle dependent fp64 operations
#pragma unroll
            for (int s = 0; s < KT; ++s) a4[s & 3] += *reinterpret_cast<const double*>(reinterpret_cast<const uint8_t*>(f1) + co[s]);
            const double a_adj = (((a4[0] + a4[1]) + (a4[2] + a4[3])) - cst) * 0.125;

            // the warp's 32 rows of the previous tile have left the staging buffer (each warp stages and stores its own rows:
            // no warpgroup-wide barrier anywhere in the loop, the four warps only meet at the a_full / mma_done mbarriers)
            if (lane == 0) bulk_wait_read0();
            __syncwarp();
            mbar_wait_wd(&mma_done[g], ((uint32_t)u) & 1u);
            tc_fence_after();
#pragma unroll
            for (int c0 = 0; c0 < 8 * KT; c0 += 32) {
                uint32_t v[32];
                double chg[4], cd[4];                  // c HG[c] and 8 c (as a double, via the 2^52 bit pattern) of the four states
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int tt = (c0 / 8 + i < KT) ? c0 / 8 + i : 0;
                    chg[i] = *reinterpret_cast<const double*>(reinterpret_cast<const uint8_t*>(g1) + co[tt]);
                    cd[i] = __hiloint2double(0x43300000, (int)co[tt]) - 4503599627370496.0;         // 8 c, exactly
                }
                tmem_ld_32x32(taddr + (uint32_t)c0, v);
                float f[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int tt = c0 / 8 + i;
                    f[i] = 0.0f;
                    if (tt < KT && (KR == 0 || tt < KR)) {
                        // exact integer sum_s (c_s - [s==t]) M_st = H 2^32 + L, both halves as doubles via the magic bits.
                        // Digits are < 2^22, so pairs combine in 32 bits; multipliers come from constant memory so that
                        // they stay IMAD / IMAD.WIDE operands instead of being strength-reduced to shifts + adds.
                        const uint32_t t01 = mad_lo(v[8 * i + 1], c_k5tc.m8, v[8 * i]);
                        const uint32_t t23 = mad_lo(v[8 * i + 3], c_k5tc.m8, v[8 * i + 2]);
                        const uint32_t t45 = mad_lo(v[8 * i + 5], c_k5tc.m8, v[8 * i + 4]);
                        const uint32_t t67 = mad_lo(v[8 * i + 7], c_k5tc.m8, v[8 * i + 6]);
                        // {t01, magic_hi} is a register pair (no instruction): L + magic = t23 2^16 + that pair
                        const unsigned long long lb = mad_wide(t23, c_k5tc.m16, ((unsigned long long)(T5_MAGIC >> 32) << 32) | t01);
                        const unsigned long long hb = mad_wide(t67, c_k5tc.m16, ((unsigned long long)(T5_MAGIC >> 32) << 32) | t45);
                        const double dl = __longlong_as_double((long long)lb);                           // L + magic
                        const double dh = __longlong_as_double((long long)hb) - 6755399441055744.0;    // H
                        // base = (H 2^32 + L) scale + A - [s==t] term, with the L part off the dependent chain of the H conversion
                        const double base = fma(dh, scale32, fma(dl, scale, a_adj)) - c_k5tc.dg[tt];
                        const double val = fma(cd[i], base, chg[i]);      // absent state: 0 * base + (+0) = +0.0 as in the reference
                        f[i] = (float)val;
                        if (WANT64 && (KR != 0 || tt < K) && bin0 + r < bins) out64[(bin0 + r) * K + tt] = val;
                    }
                }
                if constexpr (KR != 0 && KR % 2 == 0) {
                    // even row length: 8-byte stores (conflict-free at 72-byte row pitch)
                    float2* dst = reinterpret_cast<float2*>(mystage + r * KR + c0 / 8);
                    if (c0 / 8 < KR) dst[0] = make_float2(f[0], f[1]);
                    if (c0 / 8 + 2 < KR) dst[1] = make_float2(f[2], f[3]);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (c0 / 8 + i < K) mystage[r * K + c0 / 8 + i] = f[i];
                }
            }
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            if (out32 != nullptr) {
                const int wq = warp & 3;
                const long long wbin0 = bin0 + 32 * wq;
                if (t < nfull) {
                    if (lane == 0) {
                        bulk_store_1d(out32 + wbin0 * K, mystage + 32 * wq * K, (uint32_t)(32 * K * 4));
                        bulk_commit();
                    }
                } else if (wbin0 < bins) {
                    const int n = (int)((bins - wbin0) < 32 ? (bins - wbin0) : 32) * K;
                    for (int i = lane; i < n; i += 32) out32[wbin0 * K + i] = mystage[32 * wq * K + i];
                }
            }
        }
        if (lane == 0) bulk_wait0();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4 * NWG + 1) tmem_dealloc(tmem_base, 512);
}

template <int KT, int KR, int NWG, bool WANT64>
static int launch_k5_tc2(const uint16_t* cnt, int64_t bins, int K, int width, int64_t perms, const uint8_t* b_image,
                         float* o32, double* o64, cudaStream_t st) {
    constexpr int NPAD = ((8 * KT + 31) / 32) * 32;
    auto kern = k5_s2_tc_kernel<KT, KR, NWG, WANT64>;
    const size_t smem = 1024 + (size_t)NWG * T5_A_BYTES + (size_t)NPAD * 128 + (size_t)NWG * 2 * T5_BINS * K * 2 +
                        (size_t)NWG * T5_BINS * K * 4 + (size_t)(width + 2) * 16 +
                        (size_t)(6 * NWG + 1) * 8 + 16;
    EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t ntiles = (bins + T5_BINS - 1) / T5_BINS;
    kern<<<persistent_grid(ntiles, 1), NWG * 128 + 64, smem, st>>>(cnt, (long long)bins, K, width, (double)perms, b_image,
                                                                    o32, o64);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

template <int KT, int KR, int NWG>
static int launch_k5_tc(const uint16_t* cnt, int64_t bins, int K, int width, int64_t perms, const float* e, int* zero_flag,
                        float* o32, double* o64, cudaStream_t st) {
    constexpr int NPAD = ((8 * KT + 31) / 32) * 32;
    static_assert(NPAD * 128 <= sizeof(DeviceWorkspace::k5tc_b_image), "B operand image exceeds its workspace region");
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    k5tc_prepare_kernel<<<1, 256, 0, st>>>(e, K, (double)perms, NPAD, ws->k5tc_b_image, &ws->k5tc_consts, zero_flag, nullptr);
    EPI_CUDA(cudaGetLastError());
    EPI_CUDA(cudaMemcpyToSymbolAsync(c_k5tc, &ws->k5tc_consts, sizeof(K5TcConsts), 0, cudaMemcpyDeviceToDevice, st));
    if (o64 != nullptr) return launch_k5_tc2<KT, KR, NWG, true>(cnt, bins, K, width, perms, ws->k5tc_b_image, o32, o64, st);
    return launch_k5_tc2<KT, KR, NWG, false>(cnt, bins, K, width, perms, ws->k5tc_b_image, o32, o64, st);
}

// TABLE evaluation of the S2 scores on the tensor cores.  Writes *zero_flag (device int) = 1 and does nothing else when
// the expected table has a zero entry; the caller queues the DIRECT kernel behind it, gated on that flag.
int scores_s2_tc(const uint16_t* cnt, int64_t bins, int K, int width, int64_t perms, const float* e, int* zero_flag,
                 float* o32, double* o64, cudaStream_t st) {
    if (K == 18) return launch_k5_tc<18, 18, 3>(cnt, bins, K, width, perms, e, zero_flag, o32, o64, st);
    if (K == 15) return launch_k5_tc<16, 15, 4>(cnt, bins, K, width, perms, e, zero_flag, o32, o64, st);
    if (K <= 16) return launch_k5_tc<16, 0, 4>(cnt, bins, K, width, perms, e, zero_flag, o32, o64, st);
    if (K <= 18) return launch_k5_tc<18, 0, 3>(cnt, bins, K, width, perms, e, zero_flag, o32, o64, st);
    return launch_k5_tc<32, 0, 2>(cnt, bins, K, width, perms, e, zero_flag, o32, o64, st);
}

bool scores_s2_tc_eligible(int width) { return width <= T5_MAX_WIDTH; }

// the fixed-point image of -log2 E the kernel multiplies with, and F (diagnostic; used by the exactness test)
int scores_s2_tc_fixed_point(const float* e, int K, int64_t perms, unsigned long long* mfix_dev, int* fbits_host,
                             cudaStream_t st) {
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    k5tc_prepare_kernel<<<1, 256, 0, st>>>(e, K, (double)perms, 8 * EPI_MAX_STATES, ws->k5tc_b_image, &ws->k5tc_consts,
                                           &ws->prep_flags.has_zero, mfix_dev);
    EPI_CUDA(cudaGetLastError());
    K5TcConsts host;
    EPI_CUDA(cudaMemcpyAsync(&host, &ws->k5tc_consts, sizeof(host), cudaMemcpyDeviceToHost, st));
    EPI_CUDA(cudaStreamSynchronize(st));
    if (fbits_host) *fbits_host = host.fbits;
    return 0;
}

}  // namespace epi
