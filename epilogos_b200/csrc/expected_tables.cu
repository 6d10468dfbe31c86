// K2 (S1/S2 expected count tables from the per-bin counts) and K4 (normalise).
// The K2 in this file is the integer-ALU kernel; epi_expected_s1s2 runs the tensor-core Gram kernel of
// tc_tables.cu (every K <= 32) and keeps this one behind EPI_K2_ALU=1 for A/B timing and as the
// cross-check of the tests: both produce the same int64 tables bit for bit (tests/test_gpu_parity.py).
#include <stdlib.h>

#include "common.cuh"

namespace epi {

// ================================================================================================
// K2: n1[s] += sum_b c[b][s];  n2[s][t] += sum_b c[b][s]*c[b][t] - [s==t] c[b][s]
//     (expected.py:106-113 s1Calc, expected.py:146-158 s2Calc)
//
// The K x K table is cut into 6x6 blocks; only blocks on or above the diagonal are computed (the table is
// symmetric) and mirrored when they are flushed.  Each thread owns one block as 36 32-bit partial sums in
// registers and walks a private stream of bins of a shared-memory count tile: 12 LDS + 36 IMAD per bin and
// block, i.e. ~350 lane-instructions per bin at K=18 (the first version with 3x3 tiles needed ~900).
// Partials are flushed into 64-bit shared-memory atomics before they can overflow (flush_every bins),
// and once per CTA into global atomics.  Integer sums: bit-exact for any grid / flush order.
// ================================================================================================
constexpr int K2_THREADS = 256;
constexpr int K2_TILE = 512;
constexpr int K2_TS = 6;

template <int NBLK, bool FULL>     // FULL: K == 6*NBLK, no range guards on the state index
__global__ void __launch_bounds__(K2_THREADS, 2)
k2_expected_kernel(const uint16_t* __restrict__ cnt, long long bins, int K, int flush_every,
                   unsigned long long* __restrict__ n1, unsigned long long* __restrict__ n2) {
    constexpr int TS = K2_TS;
    constexpr int NPAIR = NBLK * (NBLK + 1) / 2;
    constexpr int NSTREAMS = K2_THREADS / NPAIR;

    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int tile_bytes = (K2_TILE * K * 2 + 127) & ~127;
    uint16_t* tiles[2] = {reinterpret_cast<uint16_t*>(smem_raw), reinterpret_cast<uint16_t*>(smem_raw + tile_bytes)};
    unsigned long long* s2 = reinterpret_cast<unsigned long long*>(smem_raw + 2 * tile_bytes);
    unsigned long long* s1 = s2 + K * K;
    uint64_t* full = reinterpret_cast<uint64_t*>(s1 + K);            // 2 mbarriers

    const int tid = threadIdx.x;
    const int stream_id = tid / NPAIR;
    const int pair = tid - stream_id * NPAIR;
    const bool active = stream_id < NSTREAMS;
    int bi = 0, bj = 0;
    {
        int p = pair;
        while (p >= NBLK - bi) {      // row bi of the upper triangle holds NBLK - bi blocks
            p -= NBLK - bi;
            ++bi;
        }
        bj = bi + p;
    }
    const bool diag = bi == bj;

    for (int i = tid; i < K * K + K; i += K2_THREADS) s2[i] = 0ull;   // s1 follows s2 contiguously

    uint32_t part[TS][TS];
    uint32_t partd[TS];
#pragma unroll
    for (int i = 0; i < TS; ++i) {
        partd[i] = 0;
#pragma unroll
        for (int j = 0; j < TS; ++j) part[i][j] = 0;
    }
    int pending = 0;

    auto flush = [&]() {
#pragma unroll
        for (int i = 0; i < TS; ++i) {
            const int s = bi * TS + i;
#pragma unroll
            for (int j = 0; j < TS; ++j) {
                const int q = bj * TS + j;
                if (s < K && q < K && part[i][j] != 0u) {
                    unsigned long long v = part[i][j];
                    if (diag) {
                        if (s == q) v -= partd[i];                        // c*(c-1) on the diagonal
                        if (v != 0ull) atomicAdd(&s2[s * K + q], v);
                    } else {
                        atomicAdd(&s2[s * K + q], v);
                        atomicAdd(&s2[q * K + s], v);
                    }
                }
                part[i][j] = 0;
            }
            if (diag && s < K && partd[i] != 0u) atomicAdd(&s1[s], (unsigned long long)partd[i]);
            partd[i] = 0;
        }
        pending = 0;
    };

    // Full tiles stream in through a two-deep ring of 1D bulk copies (cp.async.bulk + mbarrier); the single
    // partial tile at the end of the array is loaded cooperatively.
    const long long ntiles = (bins + K2_TILE - 1) / K2_TILE;
    const long long nfull = bins / K2_TILE;
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        mbar_fence_init();
    }
    __syncthreads();
    auto issue = [&](long long t, int buf) {
        if (t < nfull) {
            mbar_expect_tx(&full[buf], K2_TILE * K * 2);
            bulk_load_1d(tiles[buf], cnt + t * K2_TILE * K, K2_TILE * K * 2, &full[buf]);
        }
    };
    if (tid == 0) issue(blockIdx.x, 0);
    int buf = 0;
    uint32_t phase[2] = {0, 0};
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const long long bin0 = t * K2_TILE;
        const int nb = (int)((bins - bin0) < K2_TILE ? (bins - bin0) : K2_TILE);
        uint16_t* tile = tiles[buf];
        if (tid == 0) issue(t + gridDim.x, buf ^ 1);          // prefetch the next tile of this CTA
        if (t < nfull) {
            mbar_wait(&full[buf], phase[buf]);
            phase[buf] ^= 1;
        } else {
            const uint16_t* src = cnt + bin0 * K;
            for (int i = tid; i < nb * K; i += K2_THREADS) tile[i] = src[i];
            __syncthreads();
        }
        if (active) {
            for (int b = stream_id; b < nb; b += NSTREAMS) {
                const uint16_t* row = tile + b * K;
                uint32_t a[TS], c[TS];
#pragma unroll
                for (int i = 0; i < TS; ++i) {
                    const int s = bi * TS + i, q = bj * TS + i;
                    a[i] = (FULL || s < K) ? row[s] : 0u;
                    c[i] = (FULL || q < K) ? row[q] : 0u;
                }
#pragma unroll
                for (int i = 0; i < TS; ++i) {
                    partd[i] += a[i];
#pragma unroll
                    for (int j = 0; j < TS; ++j) part[i][j] += a[i] * c[j];
                }
                if (++pending >= flush_every) flush();
            }
        }
        __syncthreads();      // everyone is done with `tile` before it is refilled two iterations later
        buf ^= 1;
    }
    if (active && pending) flush();
    __syncthreads();
    for (int i = tid; i < K * K; i += K2_THREADS)
        if (n2 != nullptr && s2[i] != 0ull) atomicAdd(&n2[i], s2[i]);
    for (int i = tid; i < K; i += K2_THREADS)
        if (n1 != nullptr && s1[i] != 0ull) atomicAdd(&n1[i], s1[i]);
}

// ================================================================================================
// K4: out = float( double(N) / double(sum N) )      (expectedCombination.py:42)
// Small tables (S1: K, S2: K*K entries) are summed and divided by one CTA in one launch; large ones
// (S3: (C*K)^2 entries) use a grid-wide sum into a per-device scratch slot followed by a divide kernel.
// ================================================================================================
__device__ __forceinline__ long long block_sum_i64(long long local, long long* wsum) {
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = local;
    __syncthreads();
    long long v = 0;
    if (threadIdx.x < 32) {
        v = threadIdx.x < (blockDim.x >> 5) ? wsum[threadIdx.x] : 0;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    }
    return v;      // valid in warp 0
}

__global__ void __launch_bounds__(256) k4_small_kernel(const long long* __restrict__ counts, int n,
                                                       float* __restrict__ out) {
    __shared__ long long wsum[32];
    __shared__ double denom;
    long long local = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) local += counts[i];
    const long long total = block_sum_i64(local, wsum);
    if (threadIdx.x == 0) denom = (double)total;
    __syncthreads();
    const double d = denom;
    for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = (float)((double)counts[i] / d);
}

__global__ void __launch_bounds__(256) k4_sum_kernel(const long long* __restrict__ counts, long long n,
                                                     unsigned long long* total) {
    __shared__ long long wsum[32];
    long long local = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        local += counts[i];
    const long long v = block_sum_i64(local, wsum);
    if (threadIdx.x == 0 && v != 0) atomicAdd(total, (unsigned long long)v);
}

__global__ void __launch_bounds__(256) k4_divide_kernel(const long long* __restrict__ counts, long long n,
                                                        const unsigned long long* __restrict__ total,
                                                        float* __restrict__ out) {
    const double denom = (double)(long long)(*total);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = (float)((double)counts[i] / denom);
}

int persistent_grid(int64_t ntiles, int per_sm) {
    int64_t g = (int64_t)sm_count() * per_sm;
    if (g > ntiles) g = ntiles;
    if (g < 1) g = 1;
    return (int)g;
}

// allocated once per device: no stream-ordered malloc on the hot path
DeviceWorkspace* device_workspace() {
    static DeviceWorkspace* base[64] = {nullptr};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (base[dev] == nullptr && cudaMalloc(reinterpret_cast<void**>(&base[dev]), sizeof(DeviceWorkspace)) != cudaSuccess)
        return nullptr;
    return base[dev];
}

static unsigned long long* scratch_slot() {
    static unsigned next = 0;
    DeviceWorkspace* ws = device_workspace();
    return ws ? &ws->reduce_slots[next++ & 63] : nullptr;
}

template <int NBLK, bool FULL>
static int launch_k2_impl(const uint16_t* cnt, int64_t bins, int K, int width, int64_t* n1, int64_t* n2, cudaStream_t st) {
    const int64_t ntiles = (bins + K2_TILE - 1) / K2_TILE;
    const size_t smem = 2 * (((size_t)K2_TILE * K * 2 + 127) & ~(size_t)127) + (size_t)(K * K + K) * 8 + 16;
    auto kern = k2_expected_kernel<NBLK, FULL>;
    EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t flush_every = 0xffffffffll / ((int64_t)width * width);
    if (flush_every < 1) flush_every = 1;
    if (flush_every > (1 << 20)) flush_every = 1 << 20;
    kern<<<persistent_grid(ntiles, getenv("EPI_K2_CTAS") ? atoi(getenv("EPI_K2_CTAS")) : 2), K2_THREADS, smem, st>>>(cnt, bins, K, (int)flush_every,
                                                               reinterpret_cast<unsigned long long*>(n1),
                                                               reinterpret_cast<unsigned long long*>(n2));
    EPI_CUDA(cudaGetLastError());
    return 0;
}

template <int NBLK>
static int launch_k2(const uint16_t* cnt, int64_t bins, int K, int width, int64_t* n1, int64_t* n2, cudaStream_t st) {
    if (K == NBLK * K2_TS) return launch_k2_impl<NBLK, true>(cnt, bins, K, width, n1, n2, st);
    return launch_k2_impl<NBLK, false>(cnt, bins, K, width, n1, n2, st);
}

}  // namespace epi

using namespace epi;

extern "C" int epi_expected_s1s2(const uint16_t* cnt_dev, int64_t bins, int32_t K, int32_t width, int64_t* n1_dev,
                                 int64_t* n2_dev, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && bins < (1ll << 31), "bins=%lld out of range", (long long)bins);
    EPI_REQUIRE(K >= 1 && K <= EPI_MAX_STATES, "num_states=%d out of range [1, %d]", K, EPI_MAX_STATES);
    EPI_REQUIRE(width >= 1 && width <= 65535, "width=%d out of range [1, 65535]", width);
    if (bins == 0 || (n1_dev == nullptr && n2_dev == nullptr)) return 0;
    EPI_REQUIRE(cnt_dev != nullptr, "null count pointer");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(cnt_dev) & 15) == 0, "cnt_dev must be 16-byte aligned");
    // default: the Gram form on the tensor cores (tc_tables.cu); EPI_K2_ALU=1 selects the integer-pipe kernel (A/B timing)
    if (getenv("EPI_K2_ALU") == nullptr) return launch_k2_tc(cnt_dev, bins, K, width, n1_dev, n2_dev, st);
    if (K <= 6) return launch_k2<1>(cnt_dev, bins, K, width, n1_dev, n2_dev, st);
    if (K <= 12) return launch_k2<2>(cnt_dev, bins, K, width, n1_dev, n2_dev, st);
    if (K <= 18) return launch_k2<3>(cnt_dev, bins, K, width, n1_dev, n2_dev, st);
    if (K <= 24) return launch_k2<4>(cnt_dev, bins, K, width, n1_dev, n2_dev, st);
    return launch_k2<6>(cnt_dev, bins, K, width, n1_dev, n2_dev, st);
}

extern "C" int epi_normalize_i64(const int64_t* counts_dev, int64_t n, float* out_dev, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(n >= 0, "n=%lld negative", (long long)n);
    if (n == 0) return 0;
    EPI_REQUIRE(counts_dev != nullptr && out_dev != nullptr, "null pointer argument");
    if (n <= 16384) {
        k4_small_kernel<<<1, 256, 0, st>>>(reinterpret_cast<const long long*>(counts_dev), (int)n, out_dev);
        EPI_CUDA(cudaGetLastError());
        return 0;
    }
    unsigned long long* total = scratch_slot();
    EPI_REQUIRE(total != nullptr, "could not allocate the reduction scratch");
    EPI_CUDA(cudaMemsetAsync(total, 0, 8, st));
    int64_t blocks = (n + 256 * 8 - 1) / (256 * 8);
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    k4_sum_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const long long*>(counts_dev), n, total);
    k4_divide_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const long long*>(counts_dev), n, total,
                                                       out_dev);
    EPI_CUDA(cudaGetLastError());
    return 0;
}
