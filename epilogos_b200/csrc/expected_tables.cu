// K4 (normalise an int64 count table), the entry point of K2 (S1/S2 expected count tables from the per-bin counts: the
// tensor-core Gram kernel of tc_tables.cu) and the per-device workspace the kernels stage their small tables in.
#include "common.cuh"

namespace epi {

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
    return launch_k2_tc(cnt_dev, bins, K, n1_dev, n2_dev, st);
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
