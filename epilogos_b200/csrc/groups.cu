// Column groups of one state matrix: per-bin counts of many column subsets in one pass, and the column gather.
//
// epi_group_counts -- cnt[g][b][s] = #{ j in group g : x[b][j] == s } for every group g, reading the matrix once.
//   A CTA stages a tile of up to 128 whole rows in shared memory (cp.async, 4-byte pieces, one warp per row), then each
//   consumer thread (one bin) walks the groups' column lists, which the host padded to whole chunks: it loads the labels
//   of a chunk from its staged row (LDS.U8; the row pitch is an odd number of words, so the 32 rows a warp reads sit in 32
//   different banks) and counts them with K1's arithmetic (count_planes.cuh): one-hot words, carry-save planes, the
//   17/18-state separation and one-bit words for 19-32 states.  When a group's list ends the planes are flushed, the
//   counts unpacked, and the 32 rows of a warp leave through shared memory as 16-byte stores.  Pad entries of a list point
//   at a zero word behind the row and are kept out of state 0 as K1 keeps its zero padding out (init_counters).  No global
//   atomics; each group's block has exactly the layout epi_bin_counts writes.
//   Per-bin work is one LDS.U8 and ~4 integer instructions per listed column, so the kernel is bound by shared-memory
//   issue and the integer pipes rather than by HBM once the groups together list more columns than the matrix has.
// epi_gather_columns -- out[b][j] = x[b][idx[j]], j < n, into a 16-byte pitched matrix (pad bytes zero).
#include <vector>

#include "count_planes.cuh"

namespace epi {

constexpr int GC_THREADS = 128;              // consumer threads == rows of a full tile

// the labels of one chunk of a column list, loaded one byte per register
template <int MODE, int NB>
struct ByteSrc {
    uint32_t v[NB];
    uint32_t one;      // the value 1, opaque to the compiler so that x*one+y stays an IMAD

    template <int J>
    __device__ __forceinline__ uint32_t onehot() const {
        uint32_t sh;
        if constexpr (MODE == MODE_B1) {
            sh = v[J];
        } else {
            asm("mad.lo.u32 %0, %1, 2, 0;" : "=r"(sh) : "r"(v[J]));
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
            uint32_t t;
            asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(t) : "r"(onehot<3 * I>()), "r"(one), "r"(onehot<3 * I + 1>()));
            asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(t) : "r"(onehot<3 * I + 2>()), "r"(one), "r"(t));
            return t;
        }
    }
};

template <int MODE>
struct GroupChunk {
    static constexpr int BYTES = (MODE == MODE_B1) ? 16 : 48;        // labels per carry-save tree of 16 words
    static constexpr int FLUSH = PlaneCount<MODE>::CAP / 16;         // chunks between plane flushes
};

__device__ __forceinline__ void cp_async4(uint32_t smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}

// meta = [offsets (groups + 1)] [npad (groups)] ... [padded column lists from meta + head]; list entries are byte offsets
// into a staged row
template <int MODE>
__global__ void __launch_bounds__(GC_THREADS)
group_counts_kernel(const int8_t* __restrict__ x, long long bins, long long pitch, int row_words, int spitch, int rows,
                    const int* __restrict__ meta, int head, int groups, int num_states, uint32_t one, uint16_t* __restrict__ cnt) {
    constexpr int NP = PlaneCount<MODE>::N;
    constexpr int NACC = (MODE == MODE_B1) ? 16 : 8;
    constexpr int CH = GroupChunk<MODE>::BYTES;
    extern __shared__ __align__(16) uint8_t smem_gc[];
    uint8_t* tile = smem_gc;
    uint16_t* out_stage = reinterpret_cast<uint16_t*>(smem_gc + (((size_t)rows * spitch + 15) & ~(size_t)15));
    const int* off = meta;
    const int* npad = meta + groups + 1;
    const int* list = meta + head;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // the zero word behind every row: pad entries of the lists point at it; cp.async never writes it
    if (tid < rows) *reinterpret_cast<uint32_t*>(tile + (size_t)tid * spitch + 4 * row_words) = 0u;

    const long long ntiles = (bins + rows - 1) / rows;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const long long bin0 = t * rows;
        const int live = (int)min((long long)rows, bins - bin0);
        __syncthreads();                                            // the previous tile is consumed
        for (int r = warp; r < live; r += GC_THREADS / 32) {
            const int8_t* src = x + (bin0 + r) * pitch;
            const uint32_t dst = smem_u32(tile + (size_t)r * spitch);
            for (int w = lane; w < row_words; w += 32) cp_async4(dst + 4 * w, src + 4 * w);
        }
        asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
        __syncthreads();

        const uint8_t* row = tile + (size_t)tid * spitch;
        const bool mine = tid < live;
        for (int g = 0; g < groups; ++g) {
            uint32_t cs[EPI_MAX_STATES];
            if (mine) {
                uint32_t p[NP], acc[NACC];
#pragma unroll
                for (int k = 0; k < NP; ++k) p[k] = 0;
                init_counters(acc, npad[g]);
                uint32_t sum1 = 0, sum2 = 0;
                int pending = 0;
                const int end = off[g + 1];
                for (int j = off[g]; j < end; j += CH) {
                    ByteSrc<MODE, CH> src;
                    src.one = one;
                    const int4* l4 = reinterpret_cast<const int4*>(list + j);
#pragma unroll
                    for (int q = 0; q < CH / 4; ++q) {
                        const int4 c = __ldg(l4 + q);
                        src.v[4 * q + 0] = row[c.x];
                        src.v[4 * q + 1] = row[c.y];
                        src.v[4 * q + 2] = row[c.z];
                        src.v[4 * q + 3] = row[c.w];
                    }
                    if constexpr (MODE == MODE_F2M) {
#pragma unroll
                        for (int i = 0; i < CH; ++i) {
                            asm("mad.lo.u32 %0, %1, %2, %0;" : "+r"(sum1) : "r"(src.v[i]), "r"(one));
                            asm("mad.lo.u32 %0, %1, %1, %0;" : "+r"(sum2) : "r"(src.v[i]));
                        }
                    }
                    uint32_t carry[1] = {Tree<4>::template get<0>(src, p)};
                    Reduce<4, 1, NP>::run(carry, p);
                    if (++pending == GroupChunk<MODE>::FLUSH) {
                        flush_planes<MODE, NP, NACC>(p, acc);
                        pending = 0;
                    }
                }
                if (pending) flush_planes<MODE, NP, NACC>(p, acc);
                unpack_counts<MODE, NACC>(acc, sum1, sum2, cs);
            }
            // ---- stage the warp's 32 rows and write them with 16-byte stores when the destination allows it ----
            uint16_t* wrow = out_stage + (size_t)tid * num_states;
            if (mine) {
#pragma unroll
                for (int st = 0; st < EPI_MAX_STATES; ++st)
                    if (st < num_states) wrow[st] = (uint16_t)cs[st];
            }
            __syncwarp();
            const long long wbin0 = bin0 + warp * 32;
            const int left = live - warp * 32;
            const uint16_t* wsrc = out_stage + (size_t)warp * 32 * num_states;
            uint16_t* dst = cnt + ((long long)g * bins + wbin0) * num_states;
            if (left >= 32 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
                const int4* src16 = reinterpret_cast<const int4*>(wsrc);
                int4* dst16 = reinterpret_cast<int4*>(dst);
                for (int i = lane; i < 4 * num_states; i += 32) dst16[i] = src16[i];
            } else if (left > 0) {
                const int n = min(left, 32) * num_states;
                for (int i = lane; i < n; i += 32) dst[i] = wsrc[i];
            }
            __syncwarp();
        }
    }
}

__global__ void gather_columns_kernel(const int8_t* __restrict__ x, long long bins, long long pitch,
                                      const int* __restrict__ idx, int n, int8_t* __restrict__ out, long long out_pitch) {
    for (long long b = blockIdx.x; b < bins; b += gridDim.x) {
        const int8_t* src = x + b * pitch;
        int8_t* dst = out + b * out_pitch;
        for (int j = threadIdx.x; j < out_pitch; j += blockDim.x) dst[j] = j < n ? src[__ldg(idx + j)] : (int8_t)0;
    }
}

// host copy of a device int32 array, on the stream (the column lists are validated on the host)
static int fetch_ints(const int* dev, int64_t n, std::vector<int>& out, cudaStream_t stream) {
    out.resize((size_t)n);
    if (n == 0) return 0;
    EPI_CUDA(cudaMemcpyAsync(out.data(), dev, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, stream));
    EPI_CUDA(cudaStreamSynchronize(stream));
    return 0;
}

template <int MODE>
static int launch_group_counts(const int8_t* x, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                               const std::vector<int>& offsets, const std::vector<int>& list, int groups,
                               uint16_t* cnt, cudaStream_t stream) {
    constexpr int CH = GroupChunk<MODE>::BYTES;
    const int row_words = (cols + 3) / 4;
    int spitch = 4 * row_words + 4;                              // + the zero word
    if ((spitch / 4) % 2 == 0) spitch += 4;                      // odd words: the rows of a warp hit distinct banks
    int max_smem = 0;
    EPI_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, 0));
    const int stage_bytes = GC_THREADS * num_states * 2;
    int rows = GC_THREADS;
    while (rows > 1 && (((int64_t)rows * spitch + 15) & ~15ll) + stage_bytes > max_smem) rows -= (rows > 32 ? 32 : 1);
    const size_t smem = (((size_t)rows * spitch + 15) & ~(size_t)15) + stage_bytes;

    // meta: [offsets (groups + 1), relative to the list] [pads (groups)], then the padded lists from the first 16-byte
    // boundary on (int4 loads); pad entries point at the zero word behind the row
    const int head = (2 * groups + 1 + 3) & ~3;
    std::vector<int> meta((size_t)head, 0);
    for (int g = 0; g < groups; ++g) {
        const int n = offsets[g + 1] - offsets[g];
        const int padded = (n + CH - 1) / CH * CH;
        EPI_REQUIRE(padded <= 65535, "group %d lists %d columns: at most %d fit the 16-bit counters", g, n, 65535 / CH * CH);
        meta[g] = (int)meta.size() - head;
        meta[groups + 1 + g] = padded - n;
        meta.insert(meta.end(), list.begin() + offsets[g], list.begin() + offsets[g + 1]);
        meta.insert(meta.end(), (size_t)(padded - n), 4 * row_words);
    }
    meta[groups] = (int)meta.size() - head;

    int* meta_dev = nullptr;
    EPI_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&meta_dev), meta.size() * sizeof(int), stream));
    cudaError_t e = cudaMemcpyAsync(meta_dev, meta.data(), meta.size() * sizeof(int), cudaMemcpyHostToDevice, stream);
    int rc = 0;
    if (e != cudaSuccess) {
        set_error("cudaMemcpyAsync (group lists) failed: %s", cudaGetErrorString(e));
        rc = 1;
    } else {
        auto kern = group_counts_kernel<MODE>;
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        int per_sm = 0;
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GC_THREADS, smem);
        if (e != cudaSuccess) {
            set_error("group count kernel setup failed: %s", cudaGetErrorString(e));
            rc = 1;
        } else {
            const int64_t ntiles = (bins + rows - 1) / rows;
            int64_t grid = (int64_t)sm_count() * (per_sm > 0 ? per_sm : 1);
            if (grid > ntiles) grid = ntiles;
            kern<<<(unsigned)grid, GC_THREADS, smem, stream>>>(x, (long long)bins, (long long)pitch, row_words, spitch, rows,
                                                               meta_dev, head, groups, num_states, 1u, cnt);
            e = cudaGetLastError();
            if (e != cudaSuccess) {
                set_error("group count kernel launch failed: %s", cudaGetErrorString(e));
                rc = 1;
            }
        }
    }
    cudaFreeAsync(meta_dev, stream);
    return rc;
}

}  // namespace epi

extern "C" int epi_group_counts(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                                const int32_t* group_cols_dev, const int32_t* group_offsets_dev, int32_t groups,
                                uint16_t* cnt_dev, void* stream_) {
    using namespace epi;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && bins < (1ll << 31), "bins=%lld out of range", (long long)bins);
    EPI_REQUIRE(cols >= 1 && cols <= 65535, "cols=%d out of range [1, 65535]", cols);
    EPI_REQUIRE(pitch >= cols, "pitch=%lld smaller than cols=%d", (long long)pitch, cols);
    EPI_REQUIRE(num_states >= 1 && num_states <= EPI_MAX_STATES, "num_states=%d out of range [1, %d]", num_states,
                EPI_MAX_STATES);
    EPI_REQUIRE(groups >= 1 && groups <= EPI_MAX_GROUPS, "groups=%d out of range [1, %d]", groups, EPI_MAX_GROUPS);
    EPI_REQUIRE(group_cols_dev != nullptr && group_offsets_dev != nullptr, "null pointer argument");
    std::vector<int> offsets, list;
    if (fetch_ints(group_offsets_dev, groups + 1, offsets, stream)) return 1;
    EPI_REQUIRE(offsets[0] == 0, "group_offsets[0]=%d, must be 0", offsets[0]);
    for (int g = 0; g < groups; ++g)
        EPI_REQUIRE(offsets[g + 1] > offsets[g], "group %d is empty or its offsets decrease", g);
    if (fetch_ints(group_cols_dev, offsets[groups], list, stream)) return 1;
    for (size_t i = 0; i < list.size(); ++i)
        EPI_REQUIRE(list[i] >= 0 && list[i] < cols, "group column %d out of range [0, %d)", list[i], cols);
    if (bins == 0) return 0;
    EPI_REQUIRE(x_dev != nullptr && cnt_dev != nullptr, "null pointer argument");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(cnt_dev) & 15) == 0, "cnt_dev must be 16-byte aligned");
    const int mode = num_states <= 16 ? MODE_F2 : (num_states <= 18 ? MODE_F2M : MODE_B1);
    auto run = [&](const int8_t* x, int64_t p) {
        if (mode == MODE_F2) return launch_group_counts<MODE_F2>(x, bins, cols, p, num_states, offsets, list, groups, cnt_dev, stream);
        if (mode == MODE_F2M) return launch_group_counts<MODE_F2M>(x, bins, cols, p, num_states, offsets, list, groups, cnt_dev, stream);
        return launch_group_counts<MODE_B1>(x, bins, cols, p, num_states, offsets, list, groups, cnt_dev, stream);
    };
    if ((pitch & 15) == 0 && (reinterpret_cast<uintptr_t>(x_dev) & 15) == 0) return run(x_dev, pitch);
    // arbitrary pitch / alignment: repack on the device into a 16-byte pitched scratch matrix (as epi_bin_counts does)
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
        rc = run(scratch, pitch2);
    }
    cudaFreeAsync(scratch, stream);
    return rc;
}

extern "C" int epi_gather_columns(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, const int32_t* idx_dev,
                                  int32_t n, int8_t* out_dev, int64_t out_pitch, void* stream_) {
    using namespace epi;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && bins < (1ll << 31), "bins=%lld out of range", (long long)bins);
    EPI_REQUIRE(cols >= 1 && cols <= 65535, "cols=%d out of range [1, 65535]", cols);
    EPI_REQUIRE(pitch >= cols, "pitch=%lld smaller than cols=%d", (long long)pitch, cols);
    EPI_REQUIRE(n >= 1 && n <= 65535, "n=%d out of range [1, 65535]", n);
    EPI_REQUIRE(out_pitch >= n && (out_pitch & 15) == 0, "out_pitch=%lld must be a multiple of 16 and >= n=%d",
                (long long)out_pitch, n);
    EPI_REQUIRE(idx_dev != nullptr, "null pointer argument");
    std::vector<int> idx;
    if (fetch_ints(idx_dev, n, idx, stream)) return 1;
    for (int j = 0; j < n; ++j) EPI_REQUIRE(idx[j] >= 0 && idx[j] < cols, "column %d out of range [0, %d)", idx[j], cols);
    if (bins == 0) return 0;
    EPI_REQUIRE(x_dev != nullptr && out_dev != nullptr, "null pointer argument");
    int64_t grid = (int64_t)sm_count() * 16;
    if (grid > bins) grid = bins;
    gather_columns_kernel<<<(unsigned)grid, 256, 0, stream>>>(x_dev, (long long)bins, (long long)pitch, idx_dev, n, out_dev,
                                                               (long long)out_pitch);
    EPI_CUDA(cudaGetLastError());
    return 0;
}
