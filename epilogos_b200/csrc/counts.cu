// K1 -- per-bin state counts:  cnt[b][s] = #{ j : x[b][j] == s }
//
// Replaces np.unique(dataArr[row], return_counts=True) of the reference (expected.py:111,152;
// scores.py:341,444).  This is the only kernel that touches the bins x biosamples int8 matrix, so it is
// the HBM-bound kernel of the S1/S2 path: algorithmic traffic = `cols` bytes read per bin.
//
// Design (B200):
//  * persistent CTAs, 128 consumer threads (one bin each) + one producer warp.  The producer streams
//    [128 bins x BV*16 bytes] boxes of the matrix into a shared-memory ring with 2D TMA
//    (cp.async.bulk.tensor + mbarrier expect_tx).  The tensor map's inner extent is `cols`, so the
//    padding of the last 16-byte vector of a row and rows beyond `bins` are zero-filled by the TMA
//    unit (never read from HBM, never interpreted: the known number of zero pad bytes is kept out of
//    state 0 by the start value of its counter, init_counters).
//  * BV (16-byte vectors per box row) is odd, so consecutive rows start in different 16-byte bank
//    groups and the per-thread LDS.128 row reads are bank-conflict free without swizzling.
//  * the ALU budget at HBM speed is ~3 integer-pipe instructions per input byte, far below a
//    compare-per-state histogram (>= 9/byte).  Each label byte v becomes the "one-hot" word
//    1 << (2v mod 32) with ONE wrap-around shift (16 two-bit fields; the shifter only looks at the low
//    5 bits so no masking is needed).  Three such words are summed with one 3-input add (fields <= 3),
//    and those sums are accumulated bit-sliced with a carry-save adder tree of LOP3s (Harley-Seal):
//    ~2 LOP3 per THREE bytes.  Fields alias for states s and s+16; for 17/18-state models the two
//    aliased states are separated exactly from sum(v) and sum(v^2), which cost one IDP4A each per
//    4 bytes.  Models with more than 18 states use one-bit one-hot words (2 LOP3 per byte).
//  * counts leave through shared memory as coalesced 16-byte stores of uint16 [bins][K].
#include <utility>

#include "count_planes.cuh"

namespace epi {

constexpr int K1_ROWS = 128;                 // bins per tile == consumer threads
constexpr int K1_THREADS = K1_ROWS + 32;     // + producer warp

// Per-chunk register image of one row (the raw label words).  Pipe balance matters here: the kernel is bound
// by the integer ALU pipe (SHF/LOP3/IADD3, 64 lanes/clk/SM), while the FMA pipe (IMAD/IDP, 128 lanes/clk/SM)
// is nearly idle.  So byte extraction and the 3-way sums are expressed as IDP.4A / IMAD, which leaves
// one SHF per byte (the one-hot) and the carry-save LOP3s on the ALU pipe.
template <int BV, int MODE>
struct ChunkSrc {
    uint32_t w[4 * BV];
    uint32_t one;      // the value 1, opaque to the compiler so that x*one+y stays an IMAD

    // shift amount for byte `lane` of word `word`: 2*v (two-bit fields) or v (one-bit), possibly with
    // garbage above bit 4 for lane 0 -- the wrap-mode funnel shift reads only the low 5 bits.
    template <int J>
    __device__ __forceinline__ uint32_t onehot() const {
        constexpr int word = J >> 2, lane = J & 3;
        constexpr uint32_t mul = (MODE == MODE_B1) ? 1u : 2u;
        uint32_t sh;
        if constexpr (lane == 0) {
            sh = (MODE == MODE_B1) ? w[word] : w[word] + w[word];
        } else {
            sh = __dp4a(w[word], mul << (8 * lane), 0u);              // IDP.4A: byte `lane` times mul (FMA pipe)
        }
        uint32_t r;
        asm("shf.l.wrap.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(0u), "r"(1u), "r"(sh));
        return r;
    }
    template <int I>
    __device__ __forceinline__ uint32_t tword() const {
        if constexpr (MODE == MODE_B1) {
            return onehot<I>();
        } else {
            // two IMAD (x*1+y) instead of one IADD3: keeps the sum off the ALU pipe
            uint32_t t;
            asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(t) : "r"(onehot<3 * I>()), "r"(one), "r"(onehot<3 * I + 1>()));
            asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(t) : "r"(onehot<3 * I + 2>()), "r"(one), "r"(t));
            return t;
        }
    }
};

template <int BV, int MODE, int NP, int... G>
__device__ __forceinline__ void fold_groups(const ChunkSrc<BV, MODE>& src, uint32_t (&p)[NP],
                                            std::integer_sequence<int, G...>) {
    uint32_t carries[sizeof...(G)];
    ((carries[G] = Tree<4>::template get<G>(src, p)), ...);
    Reduce<4, sizeof...(G), NP>::run(carries, p);
}

// SW: the row is a 128-byte TMA SWIZZLE_128B row (16-byte chunk v lives at chunk v ^ swz) that holds only BV - 1 vectors;
// the last vector of the chunk is a virtual all-zero vector (label 0, part of npad).
template <int BV, int MODE, int NP, bool SW = false>
__device__ __forceinline__ void process_chunk(const uint4* __restrict__ row, uint32_t (&p)[NP], uint32_t& sum1,
                                              uint32_t& sum2, uint32_t one, int swz = 0) {
    ChunkSrc<BV, MODE> src;
    src.one = one;
#pragma unroll
    for (int v = 0; v < BV; ++v) {
        const uint4 q = SW ? (v < BV - 1 ? row[v ^ swz] : make_uint4(0u, 0u, 0u, 0u)) : row[v];
        const uint32_t qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if constexpr (MODE == MODE_F2M) {
                sum1 = __dp4a(qq[i], 0x01010101u, sum1);
                sum2 = __dp4a(qq[i], qq[i], sum2);
            }
            src.w[4 * v + i] = qq[i];
        }
    }
    constexpr int NG = (MODE == MODE_B1) ? BV : BV / 3;      // groups of 16 words
    fold_groups<BV, MODE, NP>(src, p, std::make_integer_sequence<int, NG>{});
}

// SMALL (rows of at most 128 bytes, one chunk of BV = 9 vectors, two-bit modes): the box is 128 bytes wide and written by
// the TMA unit with SWIZZLE_128B (conflict-free LDS.128 without the odd-pitch padding vector, which becomes virtual), and
// six counter planes suffice (at most 48 summed words per bin), which shortens the plane flush by a third.  For a 127-column
// matrix the per-bin fixed work (flush, unpack, staging) is as large as the per-byte work, so both count.
template <int BV, int MODE, bool SMALL = false>
__global__ void __launch_bounds__(K1_THREADS, (BV <= 9 ? 3 : 2))
k1_counts_kernel(const __grid_constant__ CUtensorMap tmap, long long bins, int nchunks, int flush_chunks, int npad,
                 int num_states, int stages, uint32_t one, uint16_t* __restrict__ cnt) {
    constexpr int NP = SMALL ? 6 : PlaneCount<MODE>::N;
    constexpr int NACC = (MODE == MODE_B1) ? 16 : 8;
    constexpr int STAGE_BYTES = (SMALL ? 8 : BV) * 16 * K1_ROWS;
    static_assert(!SMALL || (BV == 9 && MODE != MODE_B1), "the small-row variant is the one-chunk, two-bit-field case");

    extern __shared__ __align__(1024) uint8_t smem_raw_k1[];
    uint8_t* smem = SMALL ? smem_raw_k1 + ((1024u - (smem_u32(smem_raw_k1) & 1023u)) & 1023u) : smem_raw_k1;
    uint8_t* ring = smem;
    uint16_t* out_stage = reinterpret_cast<uint16_t*>(smem + (size_t)stages * STAGE_BYTES);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)stages * STAGE_BYTES +
                                                 ((K1_ROWS * num_states * 2 + 15) & ~15));
    uint64_t* empty = full + stages;

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], K1_ROWS / 32);
        }
        mbar_fence_init();
    }
    __syncthreads();

    const long long ntiles = (bins + K1_ROWS - 1) / K1_ROWS;

    if (warp == K1_ROWS / 32) {
        // ---------------- producer: one lane drives the TMA ring ----------------
        if (lane == 0) {
            tma_prefetch_desc(&tmap);
            int s = 0;
            uint32_t ph = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                for (int c = 0; c < nchunks; ++c) {
                    mbar_wait(&empty[s], ph ^ 1);
                    mbar_expect_tx(&full[s], STAGE_BYTES);
                    tma_load_2d(ring + (size_t)s * STAGE_BYTES, &tmap, c * BV * 16, (int)(tile * K1_ROWS), &full[s]);
                    if (++s == stages) {
                        s = 0;
                        ph ^= 1;
                    }
                }
            }
        }
        return;
    }

    // ---------------- consumers: one bin per thread ----------------
    int s = 0;
    uint32_t ph = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        uint32_t p[NP];
        uint32_t acc[NACC];
#pragma unroll
        for (int k = 0; k < NP; ++k) p[k] = 0;
        init_counters(acc, npad);
        uint32_t sum1 = 0, sum2 = 0;
        int pending = 0;

        for (int c = 0; c < nchunks; ++c) {
            mbar_wait(&full[s], ph);
            const uint4* row = reinterpret_cast<const uint4*>(ring + (size_t)s * STAGE_BYTES + tid * ((SMALL ? 8 : BV) * 16));
            process_chunk<BV, MODE, NP, SMALL>(row, p, sum1, sum2, one, tid & 7);
            __syncwarp();
            // p[0] is the XOR of every one-hot word of the chunk: it exists only after all of the chunk's loads returned
            if (lane == 0) mbar_arrive_after(&empty[s], p[0]);
            if (++s == stages) {
                s = 0;
                ph ^= 1;
            }
            if (++pending == flush_chunks) {
                flush_planes<MODE, NP, NACC>(p, acc);
                pending = 0;
            }
        }
        if (pending) flush_planes<MODE, NP, NACC>(p, acc);

        // ---- unpack the counters into per-state counts ----
        uint32_t cs[EPI_MAX_STATES];
        unpack_counts<MODE, NACC>(acc, sum1, sum2, cs);

        // ---- stage the warp's 32 rows and write them with 16-byte stores ----
        uint16_t* wrow = out_stage + (size_t)tid * num_states;
#pragma unroll
        for (int st = 0; st < EPI_MAX_STATES; ++st)
            if (st < num_states) wrow[st] = (uint16_t)cs[st];
        __syncwarp();
        const long long bin0 = tile * K1_ROWS + warp * 32;
        const long long left = bins - bin0;
        const uint16_t* wsrc = out_stage + (size_t)warp * 32 * num_states;
        if (left >= 32) {
            const int4* src16 = reinterpret_cast<const int4*>(wsrc);
            int4* dst16 = reinterpret_cast<int4*>(cnt + bin0 * num_states);
            for (int i = lane; i < 4 * num_states; i += 32) dst16[i] = src16[i];
        } else if (left > 0) {
            const int n = (int)left * num_states;
            for (int i = lane; i < n; i += 32) cnt[bin0 * num_states + i] = wsrc[i];
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------

struct K1Plan {
    int bv;
    int nchunks;
    int mode;
    int npad;
    bool small;      // one 128-byte swizzled box per row (see k1_counts_kernel)
};

static K1Plan plan_k1(int cols, int num_states) {
    const int nvec = (cols + 15) / 16;
    const int cand[3] = {3, 9, 15};
    int best = 3, best_total = 1 << 30;
    for (int i = 0; i < 3; ++i) {
        const int nch = (nvec + cand[i] - 1) / cand[i];
        const int total = nch * cand[i];
        if (total < best_total || (total == best_total && cand[i] > best)) {
            best = cand[i];
            best_total = total;
        }
    }
    K1Plan pl;
    pl.bv = best;
    pl.nchunks = (nvec + best - 1) / best;
    pl.mode = num_states <= 16 ? MODE_F2 : (num_states <= 18 ? MODE_F2M : MODE_B1);
    pl.npad = pl.nchunks * best * 16 - cols;
    pl.small = best == 9 && nvec <= 8 && pl.mode != MODE_B1;
    return pl;
}

template <int BV, int MODE, bool SMALL = false>
static int launch_k1(const CUtensorMap& tmap, int64_t bins, const K1Plan& pl, int num_states, uint16_t* cnt,
                          cudaStream_t stream) {
    constexpr int stage_bytes = (SMALL ? 8 : BV) * 16 * K1_ROWS;
    const int stages = (BV <= 3) ? 8 : (BV <= 9 ? 4 : 3);     // measured on B200 at 833 biosamples: 4 stages x 2 CTAs/SM: 2.22 ms;
                                              // 3 x 2: 2.26, 5 x 2: 2.26, 3 x 3: 2.32, 2 x 4: 2.35, 6 x 1: 2.79
    const int ctas_per_sm = (BV <= 3 || SMALL) ? 3 : 2;     // small rows (127 x 15): 0.470 / 0.438 / 0.465 ms at 2 / 3 / 4 CTAs per SM
    const size_t smem = (size_t)stages * stage_bytes + ((K1_ROWS * num_states * 2 + 15) & ~15) + 2 * stages * 8 +
                        (SMALL ? 1024 : 0);
    auto kern = k1_counts_kernel<BV, MODE, SMALL>;
    EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int words_per_chunk = (MODE == MODE_B1) ? 16 * BV : 16 * BV / 3;
    int flush_chunks = (SMALL ? 63 : PlaneCount<MODE>::CAP) / words_per_chunk;
    if (flush_chunks < 1) flush_chunks = 1;
    const int64_t ntiles = (bins + K1_ROWS - 1) / K1_ROWS;
    int64_t grid = (int64_t)sm_count() * ctas_per_sm;
    if (grid > ntiles) grid = ntiles;
    kern<<<(unsigned)grid, K1_THREADS, smem, stream>>>(tmap, (long long)bins, pl.nchunks, flush_chunks, pl.npad,
                                                        num_states, stages, 1u, cnt);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

template <int BV>
static int dispatch_mode(const CUtensorMap& tmap, int64_t bins, const K1Plan& pl, int num_states, uint16_t* cnt,
                         cudaStream_t stream) {
    if constexpr (BV == 9) {
        if (pl.small) {
            if (pl.mode == MODE_F2) return launch_k1<9, MODE_F2, true>(tmap, bins, pl, num_states, cnt, stream);
            return launch_k1<9, MODE_F2M, true>(tmap, bins, pl, num_states, cnt, stream);
        }
    }
    switch (pl.mode) {
        case MODE_F2: return launch_k1<BV, MODE_F2>(tmap, bins, pl, num_states, cnt, stream);
        case MODE_F2M: return launch_k1<BV, MODE_F2M>(tmap, bins, pl, num_states, cnt, stream);
        default: return launch_k1<BV, MODE_B1>(tmap, bins, pl, num_states, cnt, stream);
    }
}

int bin_counts_aligned(const int8_t* x, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states, uint16_t* cnt,
                       cudaStream_t stream) {
    const K1Plan pl = plan_k1(cols, num_states);
    tensor_map_encode_fn encode = get_tensor_map_encode();
    EPI_REQUIRE(encode != nullptr, "cuTensorMapEncodeTiled entry point not available from the driver");
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)bins};
    const cuuint64_t gstride[1] = {(cuuint64_t)pitch};
    const cuuint32_t box[2] = {(cuuint32_t)(pl.small ? 128 : pl.bv * 16), (cuuint32_t)K1_ROWS};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<int8_t*>(x), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, pl.small ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    EPI_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (cols=%d bins=%lld pitch=%lld)",
                (int)r, cols, (long long)bins, (long long)pitch);
    switch (pl.bv) {
        case 3: return dispatch_mode<3>(tmap, bins, pl, num_states, cnt, stream);
        case 9: return dispatch_mode<9>(tmap, bins, pl, num_states, cnt, stream);
        default: return dispatch_mode<15>(tmap, bins, pl, num_states, cnt, stream);
    }
}

}  // namespace epi

extern "C" int epi_bin_counts(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                              uint16_t* cnt_dev, void* stream_) {
    using namespace epi;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && bins < (1ll << 31), "bins=%lld out of range", (long long)bins);
    EPI_REQUIRE(cols >= 1 && cols <= 65535, "cols=%d out of range [1, 65535]", cols);
    EPI_REQUIRE(pitch >= cols, "pitch=%lld smaller than cols=%d", (long long)pitch, cols);
    EPI_REQUIRE(num_states >= 1 && num_states <= EPI_MAX_STATES, "num_states=%d out of range [1, %d]", num_states,
                EPI_MAX_STATES);
    if (bins == 0) return 0;
    EPI_REQUIRE(x_dev != nullptr && cnt_dev != nullptr, "null pointer argument");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(cnt_dev) & 15) == 0, "cnt_dev must be 16-byte aligned");
    if ((pitch & 15) == 0 && (reinterpret_cast<uintptr_t>(x_dev) & 15) == 0)
        return bin_counts_aligned(x_dev, bins, cols, pitch, num_states, cnt_dev, stream);
    // arbitrary pitch / alignment: repack on the device into a 16-byte pitched scratch matrix
    const int64_t pitch2 = ((int64_t)cols + 15) & ~15ll;
    int8_t* scratch = nullptr;
    EPI_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&scratch), (size_t)(pitch2 * bins), stream));
    cudaError_t e = cudaMemcpy2DAsync(scratch, (size_t)pitch2, x_dev, (size_t)pitch, (size_t)cols, (size_t)bins,
                                      cudaMemcpyDeviceToDevice, stream);
    int rc = 0;
    if (e != cudaSuccess) {
        set_error("cudaMemcpy2DAsync (repack) failed: %s", cudaGetErrorString(e));
        rc = 1;
    } else {
        rc = bin_counts_aligned(scratch, bins, cols, pitch2, num_states, cnt_dev, stream);
    }
    cudaFreeAsync(scratch, stream);
    return rc;
}
