// K7 / K8 -- paired (two-group) epilogos: shuffled-group counts, delta / null distances, quiescence mask.
//
// Reference: helpers.readStates paired-score branch (helpers.py:181-194) shuffles the labels of the combined
// [A | B] row and splits them into two halves; scores.calculateScoresPairwise (scores.py:172-256) scores
// A, B, A', B' against the shared expected table and forms
//      delta    = score(A)  - score(B)                      (float32 - float32, scores.py:223)
//      nullDiff = score(A') - score(B')                     (scores.py:224-225)
//      nullDist = sum_s nullDiff^2 * sign(sum_s nullDiff)   (float32, numpy pairwise summation, scores.py:231-232)
//      quiescent[b] = every label of A and of B equals the quiescent state (scores.py:294-303).
// S1 and S2 scores are functions of the per-bin COUNT vector only, so a shuffle is fully described by how many
// labels of each state land in A' and B'.
//
//   epi_shuffled_counts_perm    explicit permutation indices (the reference's argsort(rand) indices): used for
//                               bit-exact parity with a seeded reference run.
//   epi_shuffled_counts_philox  P independent uniform shuffles per bin drawn on the device: multivariate hypergeometric
//                               draws from the combined counts with a counter-based Philox4x32-10 stream keyed by
//                               (seed, global bin index, permutation) -- results do not depend on grid shape, on the
//                               sharding of the bins or on the GPU count.  epi_shuffled_counts_philox_range draws
//                               permutations from an offset on, so a caller can batch them.
//   epi_pairwise_combine        delta and signed squared null distance from the four float32 score arrays.
//   epi_quiescent_mask          from the group counts: cntA[q] == C1 and cntB[q] == C2.
#include "paired_draw.cuh"

namespace epi {

// ---------------------------------------------------------------- explicit permutation (test / parity mode)
__global__ void __launch_bounds__(128) shuffled_counts_perm_kernel(
    const int8_t* __restrict__ xa, long long pitch_a, int cols_a, const int8_t* __restrict__ xb, long long pitch_b,
    int cols_b, const int32_t* __restrict__ perm, long long bins, int K, int size_a, int size_b,
    uint16_t* __restrict__ out_a, uint16_t* __restrict__ out_b) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= bins) return;
    const int n = cols_a + cols_b;
    unsigned short ca[EPI_MAX_STATES], cb[EPI_MAX_STATES];
    for (int s = 0; s < EPI_MAX_STATES; ++s) ca[s] = cb[s] = 0;
    const int32_t* p = perm + b * n;
    for (int k = 0; k < size_a + size_b; ++k) {
        const int idx = p[k];
        const int v = idx < cols_a ? xa[b * pitch_a + idx] : xb[b * pitch_b + (idx - cols_a)];
        if (k < size_a) ca[v & 31]++;
        else cb[v & 31]++;
    }
    for (int s = 0; s < K; ++s) {
        out_a[b * K + s] = ca[s];
        out_b[b * K + s] = cb[s];
    }
}

// One thread per (bin, permutation); the draw is draw_shuffle (paired_draw.cuh).  The Philox stream of a draw is keyed by
// (seed; permutation = perm_offset + local index, GLOBAL bin index = bin_offset + local index): the result for a bin
// does not depend on how the bins are sharded over GPUs, on how the permutations are batched or on the launch geometry.
__global__ void __launch_bounds__(256) shuffled_counts_philox_kernel(
    const uint16_t* __restrict__ cnt_a, const uint16_t* __restrict__ cnt_b, long long bins, int K, int size_a,
    int size_b, int width, unsigned long long seed, long long bin_offset, long long perm_offset, int nperm,
    uint16_t* __restrict__ out_a, uint16_t* __restrict__ out_b) {
    extern __shared__ double lf[];                            // log(i!), i = 0..width, then 1/i, i = 0..width+1
    double* inv = lf + (width + 1);
    fill_draw_tables(lf, inv, width);
    __syncthreads();
    const long long total = bins * nperm;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long p = idx / bins, b = idx - p * bins;        // permutation-major output [P][bins][K]
        Philox rng = shuffle_stream(seed, (uint32_t)(perm_offset + p), (unsigned long long)(bin_offset + b));
        draw_shuffle(rng, cnt_a + b * K, cnt_b + b * K, K, size_a, size_b, lf, inv, [&](int s, int ga, int gb) {
            out_a[idx * K + s] = (uint16_t)ga;
            out_b[idx * K + s] = (uint16_t)gb;
        });
    }
}

// ---------------------------------------------------------------- delta / null distance
__global__ void __launch_bounds__(256) pairwise_combine_kernel(const float* __restrict__ sa, const float* __restrict__ sb,
                                                               const float* __restrict__ na, const float* __restrict__ nb,
                                                               long long rows, int K, float* __restrict__ delta,
                                                               float* __restrict__ null_dist) {
    for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < rows;
         r += (long long)gridDim.x * blockDim.x) {
        if (delta != nullptr && sa != nullptr)
            for (int s = 0; s < K; ++s) delta[r * K + s] = __fsub_rn(sa[r * K + s], sb[r * K + s]);
        if (null_dist != nullptr && na != nullptr) {
            const float* pa = na + r * K;
            const float* pb = nb + r * K;
            null_dist[r] = signed_sq_distance(K, [&](int i) { return __fsub_rn(pa[i], pb[i]); });
        }
    }
}

__global__ void __launch_bounds__(256) quiescent_mask_kernel(const uint16_t* __restrict__ cnt_a,
                                                             const uint16_t* __restrict__ cnt_b, long long bins, int K,
                                                             int cols_a, int cols_b, int q, uint8_t* __restrict__ mask) {
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < bins;
         b += (long long)gridDim.x * blockDim.x) {
        uint8_t m = 0;
        if (q >= 0 && q < K) m = (cnt_a[b * K + q] == cols_a && cnt_b[b * K + q] == cols_b) ? 1 : 0;
        mask[b] = m;
    }
}

// ---------------------------------------------------------------- real-data reductions of the paired ROI stage
// roiAndVisualPairwise.readInData (roiAndVisualPairwise.py:339-354) re-reads pairwiseDelta_*.txt.gz, i.e. it sees every
// delta after a round trip through "%.5f" text -> float64 -> float32, and computes per bin
//      distance = sum_s d^2 * sign(sum_s d)      (float32, numpy pairwise order)
//      maxDiff  = 1-based state with the largest |d|, ties -> the higher state.
// round5_text() reproduces the round trip arithmetically: the exact binary value is rounded half-even to 5 decimals
// (the residual of the scaling product is recovered with one FMA, so near-ties are decided exactly), the decimal
// q/10^5 becomes the nearest double by one correctly rounded divide (what strtod returns), then the nearest float.
__device__ __forceinline__ float round5_text(float x) {
    const double d = (double)x;
    if (!(fabs(d) < 1e9)) return x;                       // printf prints all digits; no 5-decimal rounding effect that matters
    const double ad = fabs(d);
    const double a = ad * 1e5;
    const double err = fma(ad, 1e5, -a);                  // ad*1e5 == a + err exactly
    double fl = floor(a);
    double rem = (a - fl) + err;                          // exact fractional part (|err| << 1)
    if (rem < 0.0) {
        fl -= 1.0;
        rem += 1.0;
    } else if (rem >= 1.0) {
        fl += 1.0;
        rem -= 1.0;
    }
    double q = fl;
    if (rem > 0.5 || (rem == 0.5 && fmod(fl, 2.0) != 0.0)) q += 1.0;     // round half to even
    const double r = q / 1e5;
    return (float)(signbit(d) ? -r : r);
}

__global__ void __launch_bounds__(256) pairwise_real_reduce_kernel(const float* __restrict__ delta, long long rows,
                                                                   int K, int text_round_trip,
                                                                   float* __restrict__ dist, int* __restrict__ max_diff) {
    for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < rows;
         r += (long long)gridDim.x * blockDim.x) {
        const float* p = delta + r * K;
        auto at = [&](int i) { return text_round_trip ? round5_text(p[i]) : p[i]; };
        const float sum = numpy_rowsum_f32(K, at);
        const float sq = numpy_rowsum_f32(K, [&](int i) {
            const float d = at(i);
            return __fmul_rn(d, d);
        });
        const float sign = sum > 0.f ? 1.f : (sum < 0.f ? -1.f : (sum == 0.f ? 0.f : sum));
        if (dist != nullptr) dist[r] = __fmul_rn(sq, sign);
        if (max_diff != nullptr) {
            int best = K - 1;
            float bv = fabsf(at(K - 1));
            for (int s = K - 2; s >= 0; --s) {            // argmax over the flipped row: first maximum = highest state
                const float v = fabsf(at(s));
                if (v > bv) {
                    bv = v;
                    best = s;
                }
            }
            max_diff[r] = best + 1;
        }
    }
}

}  // namespace epi

using namespace epi;

extern "C" int epi_shuffled_counts_perm(const int8_t* xa_dev, int64_t pitch_a, int32_t cols_a, const int8_t* xb_dev,
                                        int64_t pitch_b, int32_t cols_b, const int32_t* perm_dev, int64_t bins,
                                        int32_t K, int32_t size_a, int32_t size_b, uint16_t* cnt_a_out,
                                        uint16_t* cnt_b_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && cols_a >= 1 && cols_b >= 1 && K >= 1 && K <= EPI_MAX_STATES, "bad paired shape");
    EPI_REQUIRE(size_a >= 0 && size_b >= 0 && size_a + size_b <= cols_a + cols_b,
                "group sizes %d + %d exceed the %d combined biosamples", size_a, size_b, cols_a + cols_b);
    if (bins == 0) return 0;
    EPI_REQUIRE(xa_dev && xb_dev && perm_dev && cnt_a_out && cnt_b_out, "null pointer argument");
    shuffled_counts_perm_kernel<<<(unsigned)((bins + 127) / 128), 128, 0, st>>>(
        xa_dev, pitch_a, cols_a, xb_dev, pitch_b, cols_b, perm_dev, bins, K, size_a, size_b, cnt_a_out, cnt_b_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_shuffled_counts_philox_range(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins,
                                                int32_t K, int32_t width, int32_t size_a, int32_t size_b, uint64_t seed,
                                                int64_t bin_offset, int64_t perm_offset, int32_t nperm,
                                                uint16_t* cnt_a_out, uint16_t* cnt_b_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && K >= 1 && K <= EPI_MAX_STATES && nperm >= 1, "bad paired shape");
    EPI_REQUIRE(size_a >= 0 && size_b >= 0, "negative group size");
    if (int rc = check_perm_range(bin_offset, perm_offset, nperm)) return rc;
    if (bins == 0) return 0;
    EPI_REQUIRE(cnt_a_dev && cnt_b_dev && cnt_a_out && cnt_b_out, "null pointer argument");
    EPI_REQUIRE(width >= 1 && width <= 65535, "width=%d (combined biosamples) out of range [1, 65535]", width);
    if (size_a + size_b > width) {
        set_error("group sizes %d + %d exceed the %d combined biosamples", size_a, size_b, width);
        return 2;
    }
    const size_t smem = (size_t)(2 * width + 3) * 8;
    EPI_REQUIRE(smem <= 200 * 1024, "too many combined biosamples (%d) for the shuffle kernel", width);
    EPI_CUDA(cudaFuncSetAttribute(shuffled_counts_philox_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    shuffled_counts_philox_kernel<<<grid_for(bins * nperm, 256, 8), 256, smem, st>>>(
        cnt_a_dev, cnt_b_dev, bins, K, size_a, size_b, width, (unsigned long long)seed, (long long)bin_offset,
        (long long)perm_offset, nperm, cnt_a_out, cnt_b_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_shuffled_counts_philox(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins,
                                          int32_t K, int32_t width, int32_t size_a, int32_t size_b, uint64_t seed,
                                          int64_t bin_offset, int32_t nperm,
                                          uint16_t* cnt_a_out, uint16_t* cnt_b_out, void* stream_) {
    return epi_shuffled_counts_philox_range(cnt_a_dev, cnt_b_dev, bins, K, width, size_a, size_b, seed, bin_offset, 0,
                                            nperm, cnt_a_out, cnt_b_out, stream_);
}

extern "C" int epi_pairwise_combine(const float* score_a, const float* score_b, const float* null_a,
                                    const float* null_b, int64_t rows, int32_t K, float* delta_out,
                                    float* null_dist_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(rows >= 0 && K >= 1 && K <= EPI_MAX_STATES, "bad shape");
    EPI_REQUIRE((delta_out == nullptr) || (score_a && score_b), "delta needs both score arrays");
    EPI_REQUIRE((null_dist_out == nullptr) || (null_a && null_b), "null distances need both null score arrays");
    if (rows == 0) return 0;
    pairwise_combine_kernel<<<grid_for(rows, 256, 8), 256, 0, st>>>(score_a, score_b, null_a, null_b, rows, K, delta_out,
                                                                    null_dist_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_quiescent_mask(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins, int32_t K,
                                  int32_t cols_a, int32_t cols_b, int32_t quiescent_state, uint8_t* mask_out,
                                  void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && K >= 1 && K <= EPI_MAX_STATES, "bad shape");
    if (bins == 0) return 0;
    EPI_REQUIRE(cnt_a_dev && cnt_b_dev && mask_out, "null pointer argument");
    quiescent_mask_kernel<<<grid_for(bins, 256, 8), 256, 0, st>>>(cnt_a_dev, cnt_b_dev, bins, K, cols_a, cols_b,
                                                                  quiescent_state, mask_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_pairwise_real_reduce(const float* delta_dev, int64_t rows, int32_t K, int32_t text_round_trip,
                                        float* dist_out, int32_t* max_diff_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(rows >= 0 && K >= 1 && K <= EPI_MAX_STATES, "bad shape");
    if (rows == 0 || (dist_out == nullptr && max_diff_out == nullptr)) return 0;
    EPI_REQUIRE(delta_dev != nullptr, "null pointer argument");
    pairwise_real_reduce_kernel<<<grid_for(rows, 256, 8), 256, 0, st>>>(delta_dev, rows, K, text_round_trip, dist_out,
                                                                        max_diff_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}
