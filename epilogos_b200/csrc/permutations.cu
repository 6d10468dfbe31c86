// K9 -- per-bin permutation tests of paired mode: how many of P null shuffles of a bin are at least as far apart as the
// bin's real groups.
//
//   k[b] += #{ p : |null(b, p)| >= |dist[b]| },
//   null(b, p) = sum_s d_s^2 * sign(sum_s d_s),  d_s = S(A'_p)[s] - S(B'_p)[s]   (float32, numpy pairwise order)
//
// where A'_p, B'_p is shuffle p of bin b drawn by epi_shuffled_counts_philox_range (key: seed, permutation, global bin)
// and S is the run's score.  No per-(bin, permutation) value is written to memory and no atomic is taken: each bin is
// owned by one group of threads, which counts in registers and adds its total to k[b] once.
//
//   epi_null_exceedances            the counting step of the composed path: score arrays of A' and B' for a block of
//                                   permutations [n][bins][K] in, counts added into k.  With epi_shuffled_counts_philox_range
//                                   and epi_scores_s1 / epi_scores_s2 it serves every score mode (the host loops over bin
//                                   chunks x permutation blocks).
//   epi_permutation_exceedances_s1  the fused S1 path.  Per (bin, permutation) it draws the shuffle (draw_shuffle), looks
//                                   the S1 scores of A' and B' up in the K5-S1 value tables (s1_value_table, the values
//                                   epi_scores_s1 returns in TABLE mode), forms the null distance with the arithmetic of
//                                   epi_pairwise_combine and compares.  Bit-equal to the composed path.
#include "paired_draw.cuh"

namespace epi {

constexpr int K9_THREADS = 256;

__global__ void __launch_bounds__(K9_THREADS) null_exceedances_kernel(const float* __restrict__ na,
                                                                      const float* __restrict__ nb, int nperm,
                                                                      long long bins, int K,
                                                                      const float* __restrict__ dist,
                                                                      uint32_t* __restrict__ k) {
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < bins;
         b += (long long)gridDim.x * blockDim.x) {
        const float thr = fabsf(dist[b]);
        uint32_t c = 0;
        for (int p = 0; p < nperm; ++p) {
            const float* pa = na + ((long long)p * bins + b) * K;
            const float* pb = nb + ((long long)p * bins + b) * K;
            const float v = signed_sq_distance(K, [&](int i) { return __fsub_rn(pa[i], pb[i]); });
            c += fabsf(v) >= thr ? 1u : 0u;
        }
        k[b] += c;
    }
}

// T threads own one bin (group_mask); thread t takes permutations t, t + T, ...
// Shared memory: the sampler's tables (2 width + 3 doubles), then, when tables_in_smem, the value tables of A' and B'.
template <int T>
__global__ void __launch_bounds__(K9_THREADS) permutation_exceedances_s1_kernel(
    const uint16_t* __restrict__ cnt_a, const uint16_t* __restrict__ cnt_b, long long bins, int K, int size_a,
    int size_b, int width, unsigned long long seed, long long bin_offset, long long perm_offset, int nperm,
    const float* __restrict__ va_g, int wa, const float* __restrict__ vb_g, int wb, int tables_in_smem,
    const float* __restrict__ dist, uint32_t* __restrict__ k) {
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
    constexpr int GROUPS = K9_THREADS / T;
    for (long long b = blockIdx.x * (long long)GROUPS + threadIdx.x / T; b < bins; b += (long long)gridDim.x * GROUPS) {
        const float thr = fabsf(dist[b]);
        const uint16_t* ca = cnt_a + b * K;
        const uint16_t* cb = cnt_b + b * K;
        const unsigned long long gb = (unsigned long long)(bin_offset + b);
        uint32_t c = 0;
        for (int p = t; p < nperm; p += T) {
            float d[EPI_MAX_STATES];
            Philox rng = shuffle_stream(seed, (uint32_t)(perm_offset + p), gb);
            draw_shuffle(rng, ca, cb, K, size_a, size_b, lf, inv, [&](int s, int ga, int gb2) {
                d[s] = __fsub_rn(va[s * (wa + 1) + ga], vb[s * (wb + 1) + gb2]);
            });
            const float v = signed_sq_distance(K, [&](int i) { return d[i]; });
            c += fabsf(v) >= thr ? 1u : 0u;
        }
        c = group_sum<T>(gmask, c);
        if (t == 0) k[b] += c;
    }
}

}  // namespace epi

using namespace epi;

extern "C" int epi_null_exceedances(const float* null_a_dev, const float* null_b_dev, int32_t nperm, int64_t bins,
                                    int32_t K, const float* dist_dev, uint32_t* k_inout, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && nperm >= 0 && K >= 1 && K <= EPI_MAX_STATES, "bad shape");
    if (bins == 0 || nperm == 0) return 0;
    EPI_REQUIRE(null_a_dev && null_b_dev && dist_dev && k_inout, "null pointer argument");
    null_exceedances_kernel<<<grid_for(bins, K9_THREADS, 8), K9_THREADS, 0, st>>>(null_a_dev, null_b_dev, nperm, bins, K,
                                                                                  dist_dev, k_inout);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_permutation_exceedances_s1(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins,
                                              int32_t K, int32_t width, int32_t size_a, int32_t size_b, uint64_t seed,
                                              int64_t bin_offset, int64_t perm_offset, int32_t nperm,
                                              const float* exp1_dev, int32_t width_a, int32_t width_b,
                                              const float* dist_dev, uint32_t* k_inout, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && K >= 1 && K <= EPI_MAX_STATES && nperm >= 0, "bad paired shape");
    EPI_REQUIRE(size_a >= 0 && size_b >= 0, "negative group size");
    if (int rc = check_perm_range(bin_offset, perm_offset, nperm)) return rc;
    EPI_REQUIRE(width >= 1 && width <= 65535, "width=%d (combined biosamples) out of range [1, 65535]", width);
    if (size_a + size_b > width) {
        set_error("group sizes %d + %d exceed the %d combined biosamples", size_a, size_b, width);
        return 2;
    }
    // a shuffled group holds at most size labels, and its scores are looked up at count <= width_a / width_b
    EPI_REQUIRE(width_a >= size_a && width_b >= size_b && width_a >= 1 && width_b >= 1 &&
                    width_a <= S1_TABLE_MAX_WIDTH && width_b <= S1_TABLE_MAX_WIDTH,
                "score widths %d, %d must cover the group sizes %d, %d and be at most %d (the S1 value table)", width_a,
                width_b, size_a, size_b, S1_TABLE_MAX_WIDTH);
    if (bins == 0 || nperm == 0) return 0;
    EPI_REQUIRE(cnt_a_dev && cnt_b_dev && exp1_dev && dist_dev && k_inout, "null pointer argument");
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    // the float64 tables are not read here: both builds write their float64 half to the S1 scratch table
    if (int rc = s1_value_table(exp1_dev, K, width_a, ws->perm_v32[0], ws->s1_v64, st)) return rc;
    if (int rc = s1_value_table(exp1_dev, K, width_b, ws->perm_v32[1], ws->s1_v64, st)) return rc;
    const float *va = ws->perm_v32[0], *vb = ws->perm_v32[1];
    const size_t draw = (size_t)(2 * width + 3) * 8;
    const size_t tables = (size_t)K * (width_a + 1 + width_b + 1) * 4;
    // value tables in shared memory while two CTAs still fit on an SM; else they are read through L1
    const bool in_smem = draw + tables <= (size_t)110 * 1024;
    const size_t smem = draw + (in_smem ? tables : 0);
    EPI_REQUIRE(smem <= 200 * 1024, "too many combined biosamples (%d) for the shuffle kernel", width);
    return launch_fused(permutation_exceedances_s1_kernel<32>, permutation_exceedances_s1_kernel<8>,
                        permutation_exceedances_s1_kernel<1>, nperm, bins, K9_THREADS, [&](int) { return smem; }, st,
                        cnt_a_dev, cnt_b_dev, bins, K, size_a, size_b, width, (unsigned long long)seed,
                        (long long)bin_offset, (long long)perm_offset, nperm, va, width_a, vb, width_b, in_smem ? 1 : 0,
                        dist_dev, k_inout);
}
