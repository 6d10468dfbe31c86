// K11 -- stratified permutations: null shuffles that move biosample labels only within strata (tissue, donor, batch), so
// that every group keeps its own make-up in every stratum.
//
// Stratum h holds n[h][g] biosamples of group g; cnt_h [bins][K] is its count of each state over the row being shuffled.
// The shuffle of (bin b, permutation p) is draw_stratified_shuffle (paired_draw.cuh) on the stream shuffle_stream(seed,
// p, global bin): draw_multigroup_shuffle on each stratum in order, on one stream.  With one stratum it is the
// unstratified draw word for word.
//
//   epi_stratified_shuffled_counts_range  the sampler: [nperm][G][bins][K] group counts summed over the strata.  It serves
//                                         the run's own null (nperm = 1), and the composed paired (G = 2) and multi-group
//                                         permutation paths.
//   epi_stratified_exceedances_s1         the fused paired S1 path, the stratified epi_permutation_exceedances_s1: per
//                                         (bin, permutation) A' is summed over the strata in a per-thread array, B' =
//                                         (cnt_a + cnt_b) - A', both are looked up in the S1 value tables and the null
//                                         distance is compared.  Nothing per (bin, permutation) goes to memory; bit-equal
//                                         to the composed path.
#include "paired_draw.cuh"

namespace epi {

constexpr int K11_THREADS = 256;

// One thread per (bin, permutation).  Shared memory: the sampler's tables (2 width + 3 doubles, width = the widest
// stratum), the sizes [H][G], then each thread's still-needed counts, need[g * K11_THREADS + thread].
__global__ void __launch_bounds__(K11_THREADS) stratified_shuffled_counts_kernel(
    const uint16_t* __restrict__ cnt, long long hstride, int H, int G, long long bins, int K,
    const int* __restrict__ sizes_g, int width, unsigned long long seed, long long bin_offset, long long perm_offset,
    int nperm, uint16_t* __restrict__ out) {
    extern __shared__ double lf[];
    double* inv = lf + (width + 1);
    int* sz = reinterpret_cast<int*>(inv + (width + 2));
    int* need = sz + H * G + threadIdx.x;
    fill_draw_tables(lf, inv, width);
    for (int i = threadIdx.x; i < H * G; i += blockDim.x) sz[i] = sizes_g[i];
    __syncthreads();
    const long long total = bins * nperm;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long p = idx / bins, b = idx - p * bins;
        Philox rng = shuffle_stream(seed, (uint32_t)(perm_offset + p), (unsigned long long)(bin_offset + b));
        const uint16_t* c = cnt + b * K;
        uint16_t* o = out + (p * G * bins + b) * K;
        // every (state, group) is emitted once per stratum: the first stratum writes, the others add
        draw_stratified_shuffle(
            rng, H, K, G, sz, [&](int h, int s) { return (int)c[h * hstride + s]; },
            [&](int g) -> int& { return need[g * K11_THREADS]; }, lf, inv, [&](int h, int s, int g, int x) {
                uint16_t* q = o + (long long)g * bins * K + s;
                *q = (uint16_t)(h == 0 ? x : (int)*q + x);
            });
    }
}

struct PairStrata {
    int n[2 * EPI_MAX_STRATA];     // n[2 h + g]: group g's biosamples in stratum h
};

// T threads own one bin (group_mask); thread t takes permutations t, t + T, ...  Shared memory: the sampler's tables
// (2 width + 3 doubles, width = the widest stratum), then, when tables_in_smem, the value tables of A' and B'.
template <int T>
__global__ void __launch_bounds__(K11_THREADS) stratified_exceedances_s1_kernel(
    const uint16_t* __restrict__ cnt, long long hstride, int H, PairStrata sz, const uint16_t* __restrict__ cnt_a,
    const uint16_t* __restrict__ cnt_b, long long bins, int K, int width, unsigned long long seed, long long bin_offset,
    long long perm_offset, int nperm, const float* __restrict__ va_g, int wa, const float* __restrict__ vb_g, int wb,
    int tables_in_smem, const float* __restrict__ dist, uint32_t* __restrict__ k) {
    extern __shared__ double lf[];
    double* inv = lf + (width + 1);
    float* vs = reinterpret_cast<float*>(inv + (width + 2));
    const int na = K * (wa + 1), nb = K * (wb + 1);
    fill_draw_tables(lf, inv, width);
    if (tables_in_smem) {
        for (int i = threadIdx.x; i < na; i += blockDim.x) vs[i] = va_g[i];
        for (int i = threadIdx.x; i < nb; i += blockDim.x) vs[na + i] = vb_g[i];
    }
    __syncthreads();
    const float* va = tables_in_smem ? vs : va_g;
    const float* vb = tables_in_smem ? vs + na : vb_g;
    const int t = threadIdx.x % T;
    const unsigned gmask = group_mask<T>();
    constexpr int GROUPS = K11_THREADS / T;
    for (long long b = blockIdx.x * (long long)GROUPS + threadIdx.x / T; b < bins; b += (long long)gridDim.x * GROUPS) {
        const float thr = fabsf(dist[b]);
        const uint16_t* c = cnt + b * K;
        const uint16_t* ca = cnt_a + b * K;
        const uint16_t* cb = cnt_b + b * K;
        const unsigned long long gb = (unsigned long long)(bin_offset + b);
        uint32_t cnt_exceed = 0;
        for (int p = t; p < nperm; p += T) {
            int a[EPI_MAX_STATES];
            for (int s = 0; s < K; ++s) a[s] = 0;
            int need[2];
            Philox rng = shuffle_stream(seed, (uint32_t)(perm_offset + p), gb);
            draw_stratified_shuffle(
                rng, H, K, 2, sz.n, [&](int h, int s) { return (int)c[h * hstride + s]; },
                [&](int g) -> int& { return need[g]; }, lf, inv, [&](int, int s, int g, int x) {
                    if (g == 0) a[s] += x;
                });
            const float v = signed_sq_distance(K, [&](int i) {
                const int ai = a[i], bi = (int)ca[i] + (int)cb[i] - ai;
                return __fsub_rn(va[i * (wa + 1) + ai], vb[i * (wb + 1) + bi]);
            });
            cnt_exceed += fabsf(v) >= thr ? 1u : 0u;
        }
        cnt_exceed = group_sum<T>(gmask, cnt_exceed);
        if (t == 0) k[b] += cnt_exceed;
    }
}

}  // namespace epi

using namespace epi;

// checks the sizes [H][G]; returns 0 with the widest stratum and the group totals, or an error code with the message set
static int read_strata(const int32_t* sizes, int H, int G, int* width, int* totals) {
    EPI_REQUIRE(H >= 1 && H <= EPI_MAX_STRATA, "strata=%d out of range [1, %d]", H, EPI_MAX_STRATA);
    EPI_REQUIRE(G >= 2 && G <= EPI_MAX_GROUPS, "groups=%d out of range [2, %d]", G, EPI_MAX_GROUPS);
    EPI_REQUIRE(sizes != nullptr, "null pointer argument");
    long long all = 0;
    int wmax = 0;
    for (int g = 0; g < G; ++g) totals[g] = 0;
    for (int h = 0; h < H; ++h) {
        long long n = 0;
        for (int g = 0; g < G; ++g) {
            const int v = sizes[h * G + g];
            EPI_REQUIRE(v >= 0 && v <= 65535, "stratum %d holds %d biosamples of group %d", h, v, g);
            n += v;
            totals[g] += v;
        }
        EPI_REQUIRE(n >= 1, "stratum %d holds no biosample", h);
        all += n;
        if (all > 65535) break;
        wmax = n > wmax ? (int)n : wmax;
    }
    EPI_REQUIRE(all <= 65535, "more than 65535 biosamples in the strata");
    *width = wmax;
    return 0;
}

extern "C" int epi_stratified_shuffled_counts_range(const uint16_t* cnt_dev, int64_t stratum_stride, int32_t strata,
                                                    int64_t bins, int32_t num_states, const int32_t* sizes,
                                                    int32_t groups, uint64_t seed, int64_t bin_offset,
                                                    int64_t perm_offset, int32_t nperm, uint16_t* out_dev,
                                                    void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    const int K = num_states;
    EPI_REQUIRE(bins >= 0 && K >= 1 && K <= EPI_MAX_STATES, "bad stratified shape");
    EPI_REQUIRE(stratum_stride >= bins * K, "stratum stride %lld shorter than a stratum's %lld counts",
                (long long)stratum_stride, (long long)(bins * K));
    int width = 0, totals[EPI_MAX_GROUPS];
    if (int rc = read_strata(sizes, strata, groups, &width, totals)) return rc;
    if (int rc = check_perm_range(bin_offset, perm_offset, nperm)) return rc;
    if (bins == 0 || nperm == 0) return 0;
    EPI_REQUIRE(cnt_dev && out_dev, "null pointer argument");
    const size_t smem = (size_t)(2 * width + 3) * 8 + (size_t)strata * groups * 4 + (size_t)groups * K11_THREADS * 4;
    if (smem > 200 * 1024) {
        set_error("a stratum of %d biosamples (%d groups) is too wide for the shuffle kernel", width, groups);
        return 2;
    }
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    EPI_CUDA(cudaMemcpyAsync(ws->strata_sizes, sizes, (size_t)strata * groups * sizeof(int), cudaMemcpyHostToDevice, st));
    EPI_CUDA(cudaFuncSetAttribute(stratified_shuffled_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
    int per_sm = 0;
    EPI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, stratified_shuffled_counts_kernel, K11_THREADS, smem));
    stratified_shuffled_counts_kernel<<<grid_for(bins * nperm, K11_THREADS, per_sm < 1 ? 1 : per_sm), K11_THREADS, smem,
                                        st>>>(cnt_dev, (long long)stratum_stride, strata, groups, bins, K,
                                              ws->strata_sizes, width, (unsigned long long)seed, (long long)bin_offset,
                                              (long long)perm_offset, nperm, out_dev);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_stratified_exceedances_s1(const uint16_t* cnt_dev, int64_t stratum_stride, int32_t strata,
                                             const int32_t* sizes, const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev,
                                             int64_t bins, int32_t num_states, uint64_t seed, int64_t bin_offset,
                                             int64_t perm_offset, int32_t nperm, const float* exp1_dev, int32_t width_a,
                                             int32_t width_b, const float* dist_dev, uint32_t* k_inout, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    const int K = num_states;
    EPI_REQUIRE(bins >= 0 && K >= 1 && K <= EPI_MAX_STATES, "bad stratified shape");
    EPI_REQUIRE(stratum_stride >= bins * K, "stratum stride %lld shorter than a stratum's %lld counts",
                (long long)stratum_stride, (long long)(bins * K));
    int width = 0, totals[2];
    if (int rc = read_strata(sizes, strata, 2, &width, totals)) return rc;
    if (int rc = check_perm_range(bin_offset, perm_offset, nperm)) return rc;
    // a shuffled group holds its total of labels, and its scores are looked up at count <= width_a / width_b
    EPI_REQUIRE(width_a >= totals[0] && width_b >= totals[1] && width_a >= 1 && width_b >= 1 &&
                    width_a <= S1_TABLE_MAX_WIDTH && width_b <= S1_TABLE_MAX_WIDTH,
                "score widths %d, %d must cover the group sizes %d, %d and be at most %d (the S1 value table)", width_a,
                width_b, totals[0], totals[1], S1_TABLE_MAX_WIDTH);
    if (bins == 0 || nperm == 0) return 0;
    EPI_REQUIRE(cnt_dev && cnt_a_dev && cnt_b_dev && exp1_dev && dist_dev && k_inout, "null pointer argument");
    PairStrata sz;
    for (int i = 0; i < 2 * EPI_MAX_STRATA; ++i) sz.n[i] = i < 2 * strata ? sizes[i] : 0;
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    if (int rc = s1_value_table(exp1_dev, K, width_a, ws->perm_v32[0], ws->s1_v64, st)) return rc;
    if (int rc = s1_value_table(exp1_dev, K, width_b, ws->perm_v32[1], ws->s1_v64, st)) return rc;
    const float *va = ws->perm_v32[0], *vb = ws->perm_v32[1];
    const size_t draw = (size_t)(2 * width + 3) * 8;
    const size_t tables = (size_t)K * (width_a + 1 + width_b + 1) * 4;
    // value tables in shared memory while two CTAs still fit on an SM; else they are read through L1
    const bool in_smem = draw + tables <= (size_t)110 * 1024;
    const size_t smem = draw + (in_smem ? tables : 0);
    EPI_REQUIRE(smem <= 200 * 1024, "a stratum of %d biosamples is too wide for the shuffle kernel", width);
    return launch_fused(stratified_exceedances_s1_kernel<32>, stratified_exceedances_s1_kernel<8>,
                        stratified_exceedances_s1_kernel<1>, nperm, bins, K11_THREADS, [&](int) { return smem; }, st,
                        cnt_dev, (long long)stratum_stride, (int)strata, sz, cnt_a_dev, cnt_b_dev, bins, K, width,
                        (unsigned long long)seed, (long long)bin_offset, (long long)perm_offset, nperm, va, width_a, vb,
                        width_b, in_smem ? 1 : 0, dist_dev, k_inout);
}
