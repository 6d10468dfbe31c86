// Whole-genome label permutations: the per-bin counts of many column splits of one matrix, and windowed maxima of a
// per-bin statistic (the region null of paired mode and multi-group comparisons, include/epilogos_b200.h).
//
// epi_split_counts -- cnt[p][g][b][s] = #{ columns j of group g of split p : x[b][j] == s }.  A split is given by the column
//   bitsets of its first G - 1 groups; the last group is the complement.  A CTA takes a tile of 32 bins (one lane each)
//   and, once per tile, builds for every bin one bitset per PRESENT state other than the bin's most frequent one
//   (shared memory, [slot][word][bin], so the 32 lanes of a warp read 32 consecutive words).  Its 8 warps then take the
//   splits in turn; lane b of a warp counts group g of split p as sum_w popc(L_s[w] & member_g[w]) for those states (the
//   member words are the same for the whole warp: broadcast loads), derives the most frequent state as the group size
//   minus the others, and the last group as the bin's totals minus the other groups.  Per (bin, split) that is
//   (present states - 1) x ceil(N / 64) x (G - 1) AND + POPC + ADD.  Bitsets of wide matrices are taken in word chunks
//   that fit in shared memory; the counts of a chunk are added to the output, which the owning thread alone touches.
// epi_window_max -- max_inout[p] = max(max_inout[p], max_i sum_{j < W} q(stat[p][i + j])), q(x) = rint(x 2^24) in int64.
//   A CTA takes WM_TILE window starts of one row, quantises the WM_TILE + W - 1 values they read into shared memory, scans
//   them in int64 and keeps the largest difference of the scan W apart; one 64-bit atomicMax per (CTA, row).  Integer
//   sums and a maximum: the result does not depend on the tiling or on how a caller splits the rows.
#include <math.h>

#include <vector>

#include "common.cuh"

namespace epi {

constexpr int SC_TB = 32;                 // bins of a tile: one per lane
constexpr int SC_WARPS = 8;               // warps of a CTA: they share the splits
constexpr int SC_THREADS = SC_TB * SC_WARPS;

struct SplitTileMeta {
    uint32_t total[SC_TB][EPI_MAX_STATES];        // labels of every state in the bin
    uint8_t slot_state[SC_TB][EPI_MAX_STATES];    // the states that get a bitset: present, not the most frequent
    int nslot[SC_TB];
    int top[SC_TB];                                // the most frequent state (first on ties)
};

__global__ void __launch_bounds__(SC_THREADS, 1)
split_counts_kernel(const int8_t* __restrict__ x, long long bins, long long pitch, int cols, int K,
                    const unsigned long long* __restrict__ members, const int* __restrict__ sizes, int nsplit, int groups,
                    int words, int chunk_words, int max_slots, long long block_stride, uint16_t* __restrict__ cnt) {
    extern __shared__ __align__(16) uint8_t smem_sc[];
    SplitTileMeta& meta = *reinterpret_cast<SplitTileMeta*>(smem_sc);
    unsigned long long* bits = reinterpret_cast<unsigned long long*>(smem_sc + ((sizeof(SplitTileMeta) + 15) & ~(size_t)15));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long ntiles = (bins + SC_TB - 1) / SC_TB;
    const int gm = groups - 1;

    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const long long bin0 = t * SC_TB;
        const int live = (int)min((long long)SC_TB, bins - bin0);
        __syncthreads();                                            // the previous tile is done
        for (int i = tid; i < SC_TB * EPI_MAX_STATES; i += SC_THREADS) (&meta.total[0][0])[i] = 0u;
        __syncthreads();
        for (int i = tid; i < live * cols; i += SC_THREADS) {
            const int b = i / cols, j = i - b * cols;
            const int s = x[(bin0 + b) * pitch + j];
            if (s >= 0 && s < K) atomicAdd(&meta.total[b][s], 1u);
        }
        __syncthreads();
        if (tid < live) {
            int top = 0;
            for (int s = 1; s < K; ++s)
                if (meta.total[tid][s] > meta.total[tid][top]) top = s;
            int n = 0;
            for (int s = 0; s < K; ++s)
                if (s != top && meta.total[tid][s] > 0) meta.slot_state[tid][n++] = (uint8_t)s;
            meta.top[tid] = top;
            meta.nslot[tid] = n;
        }
        __syncthreads();

        for (int w0 = 0; w0 < words; w0 += chunk_words) {
            const int wc = min(chunk_words, words - w0);
            const bool first = w0 == 0;
            if (!first) __syncthreads();                            // the previous chunk's bitsets are consumed
            // ---- the chunk's bitsets: item = (slot, word, bin), bin fastest
            const int items = max_slots * wc * SC_TB;
            for (int i = tid; i < items; i += SC_THREADS) {
                const int b = i % SC_TB, jw = i / SC_TB;
                const int w = jw % wc, j = jw / wc;
                unsigned long long v = 0;
                if (b < live && j < meta.nslot[b]) {
                    const int s = meta.slot_state[b][j];
                    const int8_t* row = x + (bin0 + b) * pitch;
                    const int c0 = 64 * (w0 + w), c1 = min(c0 + 64, cols);
                    for (int c = c0; c < c1; ++c) v |= (unsigned long long)(row[c] == s) << (c - c0);
                }
                bits[i] = v;
            }
            __syncthreads();
            if (lane >= live) continue;
            const int nslot = meta.nslot[lane];
            for (int p = warp; p < nsplit; p += SC_WARPS) {
                for (int g = 0; g < gm; ++g) {
                    const unsigned long long* m = members + ((long long)p * gm + g) * words + w0;
                    uint16_t* out = cnt + ((long long)p * groups + g) * block_stride + (bin0 + lane) * K;
                    for (int j = 0; j < nslot; ++j) {
                        const unsigned long long* L = bits + (long long)j * wc * SC_TB + lane;
                        uint32_t c = 0;
                        for (int w = 0; w < wc; ++w) c += __popcll(L[(long long)w * SC_TB] & __ldg(m + w));
                        const int s = meta.slot_state[lane][j];
                        out[s] = (uint16_t)(first ? c : out[s] + c);
                    }
                }
            }
        }
        // ---- the other states: zero, the most frequent one from the group size; the last group from the totals
        if (lane >= live) continue;
        const int top = meta.top[lane], nslot = meta.nslot[lane];
        uint32_t present = 0;
        for (int j = 0; j < nslot; ++j) present |= 1u << meta.slot_state[lane][j];
        for (int p = warp; p < nsplit; p += SC_WARPS) {
            uint16_t* first_out = cnt + (long long)p * groups * block_stride + (bin0 + lane) * K;
            for (int g = 0; g < gm; ++g) {
                uint16_t* out = first_out + g * block_stride;
                uint32_t others = 0;
                for (int j = 0; j < nslot; ++j) others += out[meta.slot_state[lane][j]];
                const uint32_t size = (uint32_t)__ldg(sizes + (long long)p * groups + g);
                for (int s = 0; s < K; ++s)
                    if (!((present >> s) & 1u)) out[s] = (uint16_t)(s == top ? size - others : 0u);
            }
            for (int s = 0; s < K; ++s) {
                uint32_t r = meta.total[lane][s];
                for (int g = 0; g < gm; ++g) r -= first_out[g * block_stride + s];
                first_out[gm * block_stride + s] = (uint16_t)r;
            }
        }
    }
}

constexpr int WM_THREADS = 512;
constexpr int WM_TILE = 4096;             // window starts of a CTA

template <typename T>
__device__ __forceinline__ bool quantise(T v, long long& q) {
    const double d = (double)v;
    if (!(d >= 0.0 && d < 16777216.0)) return false;            // NaN, infinities, negatives (not -0.0), >= 2^24
    q = __double2ll_rn(ldexp(d, 24));
    return true;
}

// one CTA = (row, tile of window starts); the grid walks the (row, tile) pairs
template <typename T>
__global__ void __launch_bounds__(WM_THREADS)
window_max_kernel(const T* __restrict__ stat, long long nrows, long long row_stride, long long n, int window,
                  long long tiles, long long* __restrict__ max_inout, unsigned long long* __restrict__ bad) {
    extern __shared__ __align__(16) long long smem_wm[];
    __shared__ long long part[WM_THREADS / 32];
    __shared__ long long best_w[WM_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long starts = n - window + 1;
    for (long long blk = blockIdx.x; blk < nrows * tiles; blk += gridDim.x) {
        const long long row = blk / tiles, t0 = (blk - row * tiles) * WM_TILE;
        const int nstart = (int)min((long long)WM_TILE, starts - t0);
        const int len = nstart + window - 1;
        const T* src = stat + row * row_stride + t0;
        // ---- quantise: thread tid takes the contiguous run [tid * per, (tid + 1) * per) and scans it
        const int per = (len + WM_THREADS - 1) / WM_THREADS;
        const int a = min(len, tid * per), e = min(len, a + per);
        long long run = 0;
        for (int i = a; i < e; ++i) {
            long long q;
            if (!quantise(src[i], q)) {
                atomicMin(bad, (unsigned long long)(row * n + t0 + i));
                q = 0;
            }
            run += q;
            smem_wm[i] = run;
        }
        // ---- exclusive scan of the run totals over the CTA
        long long v = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += u;
        }
        if (lane == 31) part[warp] = v;
        __syncthreads();
        long long base = v - run;
        for (int w = 0; w < warp; ++w) base += part[w];
        for (int i = a; i < e; ++i) smem_wm[i] += base;
        __syncthreads();
        // ---- windows: S[i + W - 1] - S[i - 1]
        long long best = -1;
        for (int i = tid; i < nstart; i += WM_THREADS) {
            const long long s = smem_wm[i + window - 1] - (i > 0 ? smem_wm[i - 1] : 0ll);
            best = s > best ? s : best;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const long long u = __shfl_xor_sync(0xffffffffu, best, o);
            best = u > best ? u : best;
        }
        if (lane == 0) best_w[warp] = best;
        __syncthreads();
        if (tid == 0) {
            long long m = best_w[0];
            for (int w = 1; w < WM_THREADS / 32; ++w) m = best_w[w] > m ? best_w[w] : m;
            atomicMax(max_inout + row, m);
        }
        __syncthreads();                                            // smem and part are reused by the next (row, tile)
    }
}

}  // namespace epi

extern "C" int epi_split_counts(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                                const uint64_t* members_dev, int32_t nsplit, int32_t groups, uint16_t* cnt_dev,
                                void* stream_) {
    using namespace epi;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && bins < (1ll << 31), "bins=%lld out of range", (long long)bins);
    EPI_REQUIRE(cols >= 1 && cols <= 65535, "cols=%d out of range [1, 65535]", cols);
    EPI_REQUIRE(pitch >= cols, "pitch=%lld smaller than cols=%d", (long long)pitch, cols);
    EPI_REQUIRE(num_states >= 1 && num_states <= EPI_MAX_STATES, "num_states=%d out of range [1, %d]", num_states,
                EPI_MAX_STATES);
    EPI_REQUIRE(groups >= 2 && groups <= EPI_MAX_GROUPS, "groups=%d out of range [2, %d]", groups, EPI_MAX_GROUPS);
    EPI_REQUIRE(nsplit >= 0, "nsplit=%d is negative", nsplit);
    if (nsplit == 0) return 0;
    EPI_REQUIRE(members_dev != nullptr, "null pointer argument");
    const int words = (cols + 63) / 64;
    const int gm = groups - 1;
    // ---- the bitsets, validated on the host: no bit at or above cols, no column in two groups of a split
    std::vector<unsigned long long> mem((size_t)nsplit * gm * words);
    EPI_CUDA(cudaMemcpyAsync(mem.data(), members_dev, mem.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                             stream));
    EPI_CUDA(cudaStreamSynchronize(stream));
    const unsigned long long tail = (cols % 64) ? ~0ull << (cols % 64) : 0ull;
    std::vector<int> sizes((size_t)nsplit * groups);
    std::vector<unsigned long long> seen((size_t)words);
    for (int p = 0; p < nsplit; ++p) {
        std::fill(seen.begin(), seen.end(), 0ull);
        int used = 0;
        for (int g = 0; g < gm; ++g) {
            const unsigned long long* m = mem.data() + ((size_t)p * gm + g) * words;
            int n = 0;
            for (int w = 0; w < words; ++w) {
                EPI_REQUIRE((m[w] & seen[w]) == 0, "split %d: group %d shares column %d with an earlier group", p, g,
                            64 * w + __builtin_ctzll(m[w] & seen[w]));
                seen[w] |= m[w];
                n += __builtin_popcountll(m[w]);
            }
            EPI_REQUIRE((m[words - 1] & tail) == 0, "split %d: group %d has column %d, at or above cols=%d", p, g,
                        64 * (words - 1) + __builtin_ctzll(m[words - 1] & tail), cols);
            sizes[(size_t)p * groups + g] = n;
            used += n;
        }
        sizes[(size_t)p * groups + gm] = cols - used;
    }
    if (bins == 0) return 0;
    EPI_REQUIRE(x_dev != nullptr && cnt_dev != nullptr, "null pointer argument");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(cnt_dev) & 15) == 0, "cnt_dev must be 16-byte aligned");
    const long long block_stride = ((long long)bins * num_states + 7) & ~7ll;

    int max_smem = 0;
    EPI_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, 0));
    const size_t head = (sizeof(SplitTileMeta) + 15) & ~(size_t)15;
    const int max_slots = (num_states < cols ? num_states : cols) - 1;
    const size_t per_word = (size_t)(max_slots > 0 ? max_slots : 1) * SC_TB * 8;
    int chunk_words = (int)(((size_t)max_smem - head) / per_word);
    if (chunk_words > words) chunk_words = words;
    EPI_REQUIRE(chunk_words >= 1, "shared memory too small for one word of bitsets");
    const size_t smem = head + per_word * chunk_words;

    int* sizes_dev = nullptr;
    EPI_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&sizes_dev), sizes.size() * sizeof(int), stream));
    int rc = 0;
    cudaError_t e = cudaMemcpyAsync(sizes_dev, sizes.data(), sizes.size() * sizeof(int), cudaMemcpyHostToDevice, stream);
    const int8_t* x = x_dev;
    int64_t xp = pitch;
    int8_t* scratch = nullptr;
    if (e == cudaSuccess && ((pitch & 15) != 0 || (reinterpret_cast<uintptr_t>(x_dev) & 15) != 0)) {
        // arbitrary pitch / alignment: repack into a 16-byte pitched scratch matrix (as epi_group_counts does)
        xp = ((int64_t)cols + 15) & ~15ll;
        e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), (size_t)(xp * bins), stream);
        if (e == cudaSuccess)
            e = cudaMemcpy2DAsync(scratch, (size_t)xp, x_dev, (size_t)pitch, (size_t)cols, (size_t)bins,
                                  cudaMemcpyDeviceToDevice, stream);
        x = scratch;
    }
    if (e == cudaSuccess) e = cudaFuncSetAttribute(split_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   (int)smem);
    int per_sm = 0;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, split_counts_kernel, SC_THREADS, smem);
    if (e == cudaSuccess) {
        const int64_t ntiles = (bins + SC_TB - 1) / SC_TB;
        const int grid = persistent_grid(ntiles, per_sm > 0 ? per_sm : 1);
        split_counts_kernel<<<grid, SC_THREADS, smem, stream>>>(
            x, (long long)bins, (long long)xp, cols, num_states, reinterpret_cast<const unsigned long long*>(members_dev),
            sizes_dev, nsplit, groups, words, chunk_words, max_slots > 0 ? max_slots : 0, block_stride, cnt_dev);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
        set_error("epi_split_counts failed: %s", cudaGetErrorString(e));
        rc = 1;
    }
    if (scratch != nullptr) cudaFreeAsync(scratch, stream);
    cudaFreeAsync(sizes_dev, stream);
    return rc;
}

extern "C" int epi_window_max(const void* stat_dev, int32_t dtype, int64_t nrows, int64_t row_stride, int64_t n,
                              int32_t window, int64_t* max_inout_dev, void* stream_) {
    using namespace epi;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(dtype == 0 || dtype == 1, "dtype=%d: 0 (float32) or 1 (float64)", dtype);
    EPI_REQUIRE(nrows >= 0 && n >= 0, "nrows=%lld, n=%lld must not be negative", (long long)nrows, (long long)n);
    EPI_REQUIRE(window >= 1 && window <= 16384, "window=%d out of range [1, 16384]", window);
    EPI_REQUIRE(nrows <= 1 || row_stride >= n, "row_stride=%lld smaller than n=%lld", (long long)row_stride,
                (long long)n);
    if (nrows == 0 || n < window) return 0;
    EPI_REQUIRE(stat_dev != nullptr && max_inout_dev != nullptr, "null pointer argument");
    const long long tiles = (n - window + 1 + WM_TILE - 1) / WM_TILE;
    const size_t smem = (size_t)(WM_TILE + window - 1) * sizeof(long long);
    unsigned long long* bad = nullptr;
    EPI_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&bad), sizeof(unsigned long long), stream));
    int rc = 0;
    cudaError_t e = cudaMemsetAsync(bad, 0xff, sizeof(unsigned long long), stream);
    auto launch = [&](auto kern, const auto* stat) {
        cudaError_t r = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        int per_sm = 0;
        if (r == cudaSuccess) r = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WM_THREADS, smem);
        if (r != cudaSuccess) return r;
        const int grid = persistent_grid(nrows * tiles, per_sm > 0 ? per_sm : 1);
        kern<<<grid, WM_THREADS, smem, stream>>>(stat, (long long)nrows, (long long)row_stride, (long long)n, window,
                                                 tiles, reinterpret_cast<long long*>(max_inout_dev), bad);
        return cudaGetLastError();
    };
    if (e == cudaSuccess)
        e = dtype == 0 ? launch(window_max_kernel<float>, static_cast<const float*>(stat_dev))
                       : launch(window_max_kernel<double>, static_cast<const double*>(stat_dev));
    unsigned long long first = ~0ull;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&first, bad, sizeof(first), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {
        set_error("epi_window_max failed: %s", cudaGetErrorString(e));
        rc = 1;
    } else if (first != ~0ull) {
        const long long row = (long long)(first / (unsigned long long)n), idx = (long long)(first % (unsigned long long)n);
        double v = 0.0;
        const size_t esz = dtype == 0 ? 4 : 8;
        const char* at = static_cast<const char*>(stat_dev) + (size_t)(row * row_stride + idx) * esz;
        float f = 0.f;
        if (cudaMemcpy(dtype == 0 ? static_cast<void*>(&f) : static_cast<void*>(&v), at, esz, cudaMemcpyDeviceToHost) ==
                cudaSuccess && dtype == 0)
            v = f;
        set_error("epi_window_max: stat[%lld][%lld] = %.17g is not a finite value in [0, 2^24)", row, idx, v);
        rc = 2;
    }
    cudaFreeAsync(bad, stream);
    return rc;
}
