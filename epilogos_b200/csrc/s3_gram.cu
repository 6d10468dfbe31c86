// K3 -- S3 expected counts as an exact int8 one-hot Gram matrix on the 5th-generation tensor cores.
//
// Reference (expected.py:165-204, s3Calc): for every bin and every ORDERED pair of different biosamples
// (i, j):  N3[i][j][x[b,i]][x[b,j]] += 1.  With the one-hot matrix OH[b][j*K+s] = (x[b,j] == s) this is
//      G = OH^T OH   (CK x CK, int32),   N3[i][j][a][c] = G[i*K+a][j*K+c] for i != j,  0 for i == j.
// G is symmetric, so only tiles on or above the diagonal are computed and the rest is mirrored when the
// table is finalised (N3[j][i][c][a] = N3[i][j][a][c]).
//
//  * epi_s3_onehot   writes the TRANSPOSED one-hot OHT[m][b] (m = j*K+s, bins contiguous), which makes both
//                    GEMM operands K-major (the contraction index is the bin): the canonical TN layout.
//  * epi_s3_gram     persistent warp-specialised tcgen05 kernel on CTA pairs: 256x256 output blocks, UMMA 256x256x32
//                    (kind::i8, cta_group::2, unsigned 0/1 operands, int32 accumulators in TMEM), operands streamed by
//                    TMA (128-byte swizzle) through a 6-stage mbarrier ring; warp 0 = TMA producer, warp 1 = TMEM
//                    allocator + single-thread MMA issuer, warps 2-5 = epilogue (tcgen05.ld -> global tiles).
//                    Blocks are rasterised in column groups so the blocks in flight share operand panels in L2.
//  * epi_s3_finalize turns the (all-reduced) tile buffer into the reference's [C][C][K][K] table: int64 counts
//                    and/or float32 frequencies (float64 divide by the grand total, expectedCombination.py:42),
//                    mirroring the lower triangle and zeroing the i == j blocks.
#include "common.cuh"
#include "tc05.cuh"

namespace epi {

constexpr int G_TM = 128;           // tile rows
constexpr int G_TN = 256;           // tile cols
constexpr int G_TK = 128;           // bins per pipeline stage (= one 128-byte swizzle atom of int8)
constexpr int G_UK = 32;            // bins per tcgen05.mma (int8)
constexpr int G_THREADS = 192;
constexpr int G_GROUP = 8;          // n-tiles per raster group
constexpr int G_MAX_GROUPS = 64;

// The Gram matrix is cut into 256 x 256 blocks (Mi, nj), Mi <= nj (on or above the diagonal); block p of the schedule is
// stored as TWO 128 x 256 tiles t = 2p (rows 256 Mi .. +127) and t = 2p + 1 (rows 256 Mi + 128 .. +255), one per CTA of
// the pair that computes it.  This tile buffer is the all-reduce payload between ranks, and epi_s3_plan (its size) and
// epi_s3_finalize (the (mi, nj) -> tile look-up) count in these tiles.
struct TileSchedule {
    int mt, nt;                       // number of 128-row tiles / 256-col blocks per side
    int ngroups;
    int total;                        // tiles on or above the diagonal = 2 x blocks
    int group_count[G_MAX_GROUPS];    // blocks per raster group
};

__host__ __device__ inline int blocks_in_group(int nt, int g) {
    const int nj0 = g * G_GROUP;
    const int width = (nt - nj0) < G_GROUP ? (nt - nj0) : G_GROUP;
    int count = 0;
    for (int w = 0; w < width; ++w) count += nj0 + w + 1;          // rows Mi = 0 .. nj
    return count;
}

// block index within the schedule -> (Mi, nj); row-major inside a group of G_GROUP block columns so that consecutive blocks
// share A rows and the blocks in flight share operand panels in L2
__device__ inline void decode_block(const TileSchedule& sc, int p, int& Mi, int& nj) {
    int g = 0;
    while (g < sc.ngroups - 1 && p >= sc.group_count[g]) {
        p -= sc.group_count[g];
        ++g;
    }
    const int nj0 = g * G_GROUP;
    const int width = (sc.nt - nj0) < G_GROUP ? (sc.nt - nj0) : G_GROUP;
    for (int row = 0; row < sc.nt; ++row) {
        const int first = row > nj0 ? row - nj0 : 0;             // valid columns of this row inside the group: nj >= row
        const int valid = width - first;
        if (valid <= 0) break;
        if (p < valid) {
            Mi = row;
            nj = nj0 + first + p;
            return;
        }
        p -= valid;
    }
    Mi = 0;
    nj = nj0;      // unreachable for a consistent schedule
}

__device__ inline void decode_tile(const TileSchedule& sc, int t, int& mi, int& nj) {
    int Mi;
    decode_block(sc, t >> 1, Mi, nj);
    mi = 2 * Mi + (t & 1);
}

// ================================================================================================
// one-hot expansion, transposed:  OHT[(j*K+s)][b] = (x[b][j] == s)
// CTA = 128 bins x 32 biosamples.  Labels are staged transposed in shared memory, then every thread
// produces 16-byte (16-bin) segments of output rows with byte-parallel compares.
// ================================================================================================
constexpr int OH_BINS = 128;
constexpr int OH_COLS = 32;

__global__ void __launch_bounds__(256) s3_onehot_kernel(const int8_t* __restrict__ x, long long bins, int cols,
                                                        long long pitch, int K, int8_t* __restrict__ oht,
                                                        long long bp) {
    __shared__ __align__(16) uint8_t xs[OH_COLS][OH_BINS + 16];
    const long long b0 = (long long)blockIdx.x * OH_BINS;
    const int j0 = blockIdx.y * OH_COLS;
    const int tid = threadIdx.x;
    // load [128 bins][32 cols] and transpose into xs[col][bin]; out-of-range -> 0xFF (matches no state)
    for (int i = tid; i < OH_BINS * OH_COLS; i += 256) {
        const int b = i / OH_COLS, j = i - b * OH_COLS;
        uint8_t v = 0xFF;
        if (b0 + b < bins && j0 + j < cols) v = (uint8_t)x[(b0 + b) * pitch + j0 + j];
        xs[j][b] = v;
    }
    __syncthreads();
    const int ncol = (cols - j0) < OH_COLS ? (cols - j0) : OH_COLS;
    const int nrows = ncol * K;                       // output rows of this CTA
    // 8 threads cover one 128-byte row segment (16 bytes each)
    for (int r = tid >> 3; r < nrows; r += 32) {
        const int j = r / K, s = r - j * K;
        const int seg = tid & 7;
        const uint4 q = *reinterpret_cast<const uint4*>(&xs[j][seg * 16]);
        const uint32_t pat = (uint32_t)s * 0x01010101u;
        uint4 o;
        o.x = __vcmpeq4(q.x, pat) & 0x01010101u;
        o.y = __vcmpeq4(q.y, pat) & 0x01010101u;
        o.z = __vcmpeq4(q.z, pat) & 0x01010101u;
        o.w = __vcmpeq4(q.w, pat) & 0x01010101u;
        *reinterpret_cast<uint4*>(oht + ((long long)(j0 + j) * K + s) * bp + b0 + seg * 16) = o;
    }
}

// ================================================================================================
// Gram kernel: a CTA pair (cluster of 2 = one TPC) computes one 256 x 256 block with
// tcgen05.mma.cta_group::2 (UMMA 256 x 256 x 32).  CTA r of the pair stages rows 256 Mi + 128 r .. +127 of the A operand
// and rows 256 nj + 128 r .. +127 of the B operand -- 32 KB per 128-bin stage instead of the 48 KB (128 A rows + 256 B
// rows) of a one-CTA 128 x 256 tile.  A one-CTA kernel reached 3.2 POP/s, bound by operand delivery from L2 (94 B/clk/SM
// at tensor peak), not by the tensor pipe (4.47 POP/s with operand loads disabled).  Two 256-column accumulators per CTA
// (all 512 TMEM columns) let the epilogue of block p overlap the MMAs of block p + 1.
//   warp 0: TMA producer (both CTAs; transaction bytes of both land on the LEADER's full barrier)
//   warp 1: TMEM allocator (both CTAs) + single-thread MMA issuer (leader CTA only; commits are multicast to both CTAs)
//   warps 2-5: epilogue, each CTA drains its own 128 accumulator rows into its tile of the block
// ================================================================================================
constexpr int G2_STAGES = 6;
constexpr int G2_HALF_BYTES = 128 * G_TK;               // 128 rows x 128 bins = 16 KB
constexpr int G2_STAGE_BYTES = 2 * G2_HALF_BYTES;       // A half + B half per CTA
constexpr uint32_t G2_PEER_MASK = 0xFEFFFFFFu;          // shared::cluster address of the same offset in CTA 0 of the pair
constexpr uint32_t G2_IDESC = umma_i8_idesc(256, 256);

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA 0 of the pair (works from either CTA)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & G2_PEER_MASK) : "memory");
}
// 2D tiled TMA load whose completion bytes are counted on the LEADER CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar) & G2_PEER_MASK)
        : "memory");
}
__device__ __forceinline__ void umma2_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}
// mbarriers at this offset in BOTH CTAs arrive once all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma2_commit_both(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((unsigned short)3)
                 : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G_THREADS, 1)
s3_gram2_kernel(const __grid_constant__ CUtensorMap map, const __grid_constant__ TileSchedule sched, int kblocks,
                int accumulate, int probe, int32_t* __restrict__ tiles) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* ring = smem;                                                             // G2_STAGES * 32 KB
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + G2_STAGES * G2_STAGE_BYTES);  // TMA (both CTAs) -> MMA, leader's copy
    uint64_t* empty = full + G2_STAGES;                                               // MMA -> TMA, one copy per CTA
    uint64_t* tmem_full = empty + G2_STAGES;                                          // [2] MMA -> epilogue, one copy per CTA
    uint64_t* tmem_empty = tmem_full + 2;                                             // [2] epilogues of both CTAs -> MMA, leader's copy
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int nblocks = sched.total >> 1;
    const int first = blockIdx.x >> 1, stride = gridDim.x >> 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < G2_STAGES; ++s) {
            mbar_init(&full[s], 2);            // the leader's expect_tx arrive + the peer producer's arrive
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full[a], 1);
            mbar_init(&tmem_empty[a], 8);      // four epilogue warps of each CTA
        }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc2(tmem_slot, 512);        // two 256-column accumulators x 128 lanes in each CTA
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------ TMA producer (both CTAs) ------------------------------
        if (lane == 0) {
            tma_prefetch_desc(&map);
            int s = 0;
            uint32_t ph = 0;
            long long issued = 0;
            for (int p = first; p < nblocks; p += stride) {
                int Mi, nj;
                decode_block(sched, p, Mi, nj);
                const int a_row = (2 * Mi + (int)rank) * 128, b_row = nj * 256 + (int)rank * 128;
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait_spin_wd(&empty[s], ph ^ 1);
                    const bool load = !(probe && issued >= G2_STAGES);
                    if (leader) {
                        if (load) mbar_expect_tx(&full[s], 2 * G2_STAGE_BYTES);
                        else mbar_arrive(&full[s]);
                    } else {
                        mbar_arrive_leader(&full[s]);
                    }
                    if (load) {
                        uint8_t* st = ring + s * G2_STAGE_BYTES;
                        tma_load_2d_2sm(st, &map, kb * G_TK, a_row, &full[s]);
                        tma_load_2d_2sm(st + G2_HALF_BYTES, &map, kb * G_TK, b_row, &full[s]);
                    }
                    ++issued;
                    if (++s == G2_STAGES) {
                        s = 0;
                        ph ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------ MMA issuer (one thread of the leader CTA) ------------------------------
        if (lane == 0 && leader) {
            int s = 0, acc = 0;
            uint32_t ph = 0, acc_ph[2] = {0u, 0u};
            for (int p = first; p < nblocks; p += stride) {
                mbar_wait_spin_wd(&tmem_empty[acc], acc_ph[acc] ^ 1);        // both CTAs have drained this accumulator
                tc_fence_after();
                const uint32_t d = tmem_base + (uint32_t)(acc * 256);
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait_spin_wd(&full[s], ph);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(ring + s * G2_STAGE_BYTES);
                    const uint64_t a_desc = make_kmajor_sw128_desc(a_addr);
                    const uint64_t b_desc = make_kmajor_sw128_desc(a_addr + G2_HALF_BYTES);
#pragma unroll
                    for (int k = 0; k < G_TK / G_UK; ++k)
                        umma2_i8(d, a_desc + 2 * k, b_desc + 2 * k, G2_IDESC, (kb | k) != 0 ? 1u : 0u);
                    umma2_commit_both(&empty[s]);             // the stage may be refilled in both CTAs
                    if (++s == G2_STAGES) {
                        s = 0;
                        ph ^= 1;
                    }
                }
                umma2_commit_both(&tmem_full[acc]);           // accumulator complete, in both CTAs
                acc_ph[acc] ^= 1;
                acc ^= 1;
            }
        }
    } else {
        // ------------------------------ epilogue: own 128 accumulator rows -> own tile of the block ------------------------------
        const int quarter = warp & 3;
        int acc = 0;
        uint32_t acc_ph[2] = {0u, 0u};
        for (int p = first; p < nblocks; p += stride) {
            mbar_wait_spin_wd(&tmem_full[acc], acc_ph[acc]);
            acc_ph[acc] ^= 1;
            tc_fence_after();
            const long long t = 2ll * p + rank;
            int32_t* dst = tiles + t * (G_TM * G_TN) + (long long)(quarter * 32 + lane) * G_TN;
#pragma unroll 1
            for (int c0 = 0; c0 < G_TN; c0 += 32) {
                uint32_t v[32];
                tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 256 + c0), v);
                int4* d4 = reinterpret_cast<int4*>(dst + c0);
                if (accumulate) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        int4 o = d4[i];
                        o.x += (int)v[4 * i];
                        o.y += (int)v[4 * i + 1];
                        o.z += (int)v[4 * i + 2];
                        o.w += (int)v[4 * i + 3];
                        d4[i] = o;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        d4[i] = make_int4((int)v[4 * i], (int)v[4 * i + 1], (int)v[4 * i + 2], (int)v[4 * i + 3]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
            acc ^= 1;
        }
    }
    tc_fence_before();
    cluster_sync_all();
    if (warp == 1) tmem_dealloc2(tmem_base, 512);
}

// ================================================================================================
// finalise: tile buffer -> [C][C][K][K] int64 counts and / or float32 frequencies
// one thread per output element (i, j, a, c); reads G[min][max] from the tile that holds it
// ================================================================================================
__global__ void __launch_bounds__(256) s3_finalize_kernel(const int32_t* __restrict__ tiles, TileSchedule sched,
                                                          const int* __restrict__ tile_index, int cols, int K,
                                                          double total, long long* __restrict__ counts,
                                                          float* __restrict__ expf) {
    const long long n = (long long)cols * cols * K * K;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % K);
        long long r = idx / K;
        const int a = (int)(r % K);
        r /= K;
        const int j = (int)(r % cols);
        const int i = (int)(r / cols);
        long long v = 0;
        if (i != j) {
            int m = i * K + a, q = j * K + c;                 // G[m][q] == G[q][m]
            if (m > q) {
                const int tmp = m;
                m = q;
                q = tmp;
            }
            const int mi = m / G_TM, nj = q / G_TN;
            const int t = tile_index[mi * sched.nt + nj];
            v = tiles[(long long)t * (G_TM * G_TN) + (long long)(m - mi * G_TM) * G_TN + (q - nj * G_TN)];
        }
        if (counts != nullptr) counts[idx] = v;
        if (expf != nullptr) expf[idx] = (float)((double)v / total);
    }
}

__global__ void s3_tile_index_kernel(TileSchedule sched, int* __restrict__ tile_index) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < sched.total; t += gridDim.x * blockDim.x) {
        int mi, nj;
        decode_tile(sched, t, mi, nj);
        tile_index[mi * sched.nt + nj] = t;
    }
}

static TileSchedule make_schedule(int64_t mp) {
    TileSchedule sc;
    memset(&sc, 0, sizeof(sc));
    sc.mt = (int)(mp / G_TM);
    sc.nt = (int)(mp / G_TN);
    sc.ngroups = (sc.nt + G_GROUP - 1) / G_GROUP;
    sc.total = 0;
    for (int g = 0; g < sc.ngroups; ++g) {
        sc.group_count[g] = blocks_in_group(sc.nt, g);
        sc.total += 2 * sc.group_count[g];
    }
    return sc;
}

static int make_oht_map(CUtensorMap* map, const int8_t* oht, int64_t mp, int64_t bp, int box_rows) {
    tensor_map_encode_fn encode = get_tensor_map_encode();
    EPI_REQUIRE(encode != nullptr, "cuTensorMapEncodeTiled entry point not available from the driver");
    const cuuint64_t gdim[2] = {(cuuint64_t)bp, (cuuint64_t)mp};
    const cuuint64_t gstride[1] = {(cuuint64_t)bp};
    const cuuint32_t box[2] = {(cuuint32_t)G_TK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<int8_t*>(oht), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    EPI_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (one-hot operand) failed with CUresult %d", (int)r);
    return 0;
}

}  // namespace epi

using namespace epi;

extern "C" int epi_s3_plan(int64_t bins, int32_t cols, int32_t K, int64_t* mp, int64_t* bp, int64_t* ntiles,
                           int64_t* onehot_bytes, int64_t* tile_bytes) {
    EPI_REQUIRE(bins >= 0 && cols >= 1 && K >= 1 && K <= EPI_MAX_STATES, "bad S3 shape");
    const int64_t m = (((int64_t)cols * K + G_TN - 1) / G_TN) * G_TN;
    const int64_t b = ((bins + G_TK - 1) / G_TK) * G_TK;
    EPI_REQUIRE(m / G_TN <= (int64_t)G_MAX_GROUPS * G_GROUP, "biosamples x states = %lld is too large for the S3 tile schedule",
                (long long)cols * K);
    const TileSchedule sc = make_schedule(m);
    if (mp) *mp = m;
    if (bp) *bp = b;
    if (ntiles) *ntiles = sc.total;
    if (onehot_bytes) *onehot_bytes = m * b;
    if (tile_bytes) *tile_bytes = (int64_t)sc.total * G_TM * G_TN * 4 + (int64_t)sc.mt * sc.nt * 4;
    return 0;
}

extern "C" int epi_s3_onehot(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t K,
                             int8_t* oht_dev, int64_t mp, int64_t bp, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 1 && cols >= 1 && pitch >= cols && K >= 1 && K <= EPI_MAX_STATES, "bad S3 shape");
    EPI_REQUIRE(mp >= (int64_t)cols * K && mp % G_TN == 0 && bp >= bins && bp % G_TK == 0,
                "mp / bp must come from epi_s3_plan");
    EPI_REQUIRE(x_dev != nullptr && oht_dev != nullptr, "null pointer argument");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(oht_dev) & 127) == 0, "oht_dev must be 128-byte aligned");
    // padding rows [cols*K, mp) and padding bins are zero
    EPI_CUDA(cudaMemsetAsync(oht_dev + (int64_t)cols * K * bp, 0, (size_t)((mp - (int64_t)cols * K) * bp), st));
    dim3 grid((unsigned)(bp / OH_BINS), (unsigned)((cols + OH_COLS - 1) / OH_COLS));
    s3_onehot_kernel<<<grid, 256, 0, st>>>(x_dev, bins, cols, pitch, K, oht_dev, bp);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_s3_gram(const int8_t* oht_dev, int64_t mp, int64_t bp, int32_t* tiles_dev, int32_t accumulate,
                           void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(mp >= G_TN && mp % G_TN == 0 && bp >= G_TK && bp % G_TK == 0, "mp / bp must come from epi_s3_plan");
    EPI_REQUIRE(bp / G_TK < (1ll << 31) && bp < (1ll << 31), "too many bins for one launch: chunk the bins");
    EPI_REQUIRE(oht_dev != nullptr && tiles_dev != nullptr, "null pointer argument");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(tiles_dev) & 15) == 0, "tiles_dev must be 16-byte aligned");
    const TileSchedule sc = make_schedule(mp);
    const int probe = (accumulate & 2) ? 1 : 0;      // bit 1 of `accumulate`: tensor-peak probe (results are garbage)
    // one tensor map with 128-row boxes serves the A and the B halves
    CUtensorMap map;
    if (int rc = make_oht_map(&map, oht_dev, mp, bp, 128)) return rc;
    const size_t smem = (size_t)G2_STAGES * G2_STAGE_BYTES + (2 * G2_STAGES + 4) * 8 + 16 + 1024;
    EPI_CUDA(cudaFuncSetAttribute(s3_gram2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count() & ~1;
    if (grid > sc.total) grid = sc.total;              // total is even: two CTAs per block
    s3_gram2_kernel<<<grid, G_THREADS, smem, st>>>(map, sc, (int)(bp / G_TK), accumulate & 1, probe, tiles_dev);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_s3_finalize(int32_t* tiles_dev, int32_t cols, int32_t K, int64_t mp, int64_t total_bins,
                               int64_t* counts_dev, float* exp_dev, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(cols >= 1 && K >= 1 && mp >= (int64_t)cols * K && mp % G_TN == 0, "bad S3 shape");
    EPI_REQUIRE(tiles_dev != nullptr, "null pointer argument");
    if (counts_dev == nullptr && exp_dev == nullptr) return 0;
    const TileSchedule sc = make_schedule(mp);
    // the (mi, nj) -> tile lookup lives right after the tiles in the workspace sized by epi_s3_plan
    int* tile_index = reinterpret_cast<int*>(tiles_dev + (int64_t)sc.total * G_TM * G_TN);
    s3_tile_index_kernel<<<(sc.total + 255) / 256, 256, 0, st>>>(sc, tile_index);
    const double total = (double)total_bins * (double)cols * (double)(cols - 1);      // sum of the table (exact)
    const int64_t n = (int64_t)cols * cols * K * K;
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    s3_finalize_kernel<<<(unsigned)blocks, 256, 0, st>>>(tiles_dev, sc, tile_index, cols, K, total,
                                                         reinterpret_cast<long long*>(counts_dev), exp_dev);
    EPI_CUDA(cudaGetLastError());
    return 0;
}
