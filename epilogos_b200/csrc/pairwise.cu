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
//                               sharding of the bins or on the GPU count.
//   epi_pairwise_combine        delta and signed squared null distance from the four float32 score arrays.
//   epi_quiescent_mask          from the group counts: cntA[q] == C1 and cntB[q] == C2.
#include "common.cuh"

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

// Hypergeometric variate by inversion from the mode (zig-zag search): number of "successes" among n draws without
// replacement from a population of N holding K successes.  Everything is float64: the uniform has 53 random bits (two
// Philox words), pmf(mode) comes from a shared-memory table of log(i!), the pmf ratios of the walk are products of exact
// integers with a shared-memory table of reciprocals 1/i (relative error ~1e-16 per step), so every outcome whose
// probability exceeds ~1e-16 is reachable with its own probability -- the resolution of the reference's
// argsort(np.random.rand(...)) shuffle, whose uniforms carry 53 bits as well (helpers.py:183).  The walk visits
// O(standard deviation) values; it can run out of outcomes only through accumulated rounding (total mass 1 - O(1e-13)),
// and then the residual goes to the last outcome visited on the heavier side.  Used per state instead of walking every
// label of the row (6x fewer operations than per-label selection sampling at 833 biosamples).
__device__ __forceinline__ double uniform53(Philox& rng) {
    const uint32_t hi = rng.next(), lo = rng.next();
    // (0, 1): 53 random bits + one half
    return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6) + 0.5) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ int hypergeometric(Philox& rng, int N, int K, int n, const double* __restrict__ lf,
                                              const double* __restrict__ inv) {
    const int lo = max(0, n - (N - K)), hi = min(n, K);
    if (lo >= hi) return lo;
    int mode = (int)(((long long)(n + 1) * (K + 1)) / (N + 2));
    mode = min(max(mode, lo), hi);
    const double logp = (lf[K] - lf[mode] - lf[K - mode]) + (lf[N - K] - lf[n - mode] - lf[N - K - n + mode]) -
                        (lf[N] - lf[n] - lf[N - n]);
    const double pm = exp(logp);
    double u = uniform53(rng) - pm;
    if (u <= 0.0) return mode;
    int xu = mode, xd = mode;
    double pu = pm, pd = pm;
    const int off = N - K - n;                       // may be negative; off + x >= 0 for every feasible x
    for (;;) {
        const bool can_up = xu < hi, can_dn = xd > lo;
        if (!can_up && !can_dn) return pu >= pd ? xu : xd;     // rounding residue (~1e-13 of the mass)
        if (can_up) {
            // p(x+1)/p(x) = (K-x)(n-x) / ((x+1)(N-K-n+x+1)): integer products are exact in float64
            pu *= ((double)(K - xu) * (double)(n - xu)) * (inv[xu + 1] * inv[off + xu + 1]);
            ++xu;
            u -= pu;
            if (u <= 0.0) return xu;
        }
        if (can_dn) {
            // p(x-1)/p(x) = x (N-K-n+x) / ((K-x+1)(n-x+1))
            pd *= ((double)xd * (double)(off + xd)) * (inv[K - xd + 1] * inv[n - xd + 1]);
            --xd;
            u -= pd;
            if (u <= 0.0) return xd;
        }
    }
}

// One thread per (bin, permutation).  A uniform shuffle of the combined row split into A' (size_a labels) and
// B' (size_b labels) is, for count-based scores, a multivariate hypergeometric draw: walking over the states,
//   a'_s ~ HG(remaining labels, c_s, still needed by A'),  b'_s ~ HG(remaining - needed by A', c_s - a'_s, needed by B').
// The Philox stream of a draw is keyed by (seed; permutation, GLOBAL bin index = bin_offset + local index): the result
// for a bin does not depend on how the bins are sharded over GPUs or on the launch geometry.
__global__ void __launch_bounds__(256) shuffled_counts_philox_kernel(
    const uint16_t* __restrict__ cnt_a, const uint16_t* __restrict__ cnt_b, long long bins, int K, int size_a,
    int size_b, int width, unsigned long long seed, long long bin_offset, int nperm, uint16_t* __restrict__ out_a,
    uint16_t* __restrict__ out_b) {
    extern __shared__ double lf[];                            // log(i!), i = 0..width, then 1/i, i = 0..width+1
    double* inv = lf + (width + 1);
    for (int i = threadIdx.x; i <= width; i += blockDim.x) lf[i] = lgamma((double)i + 1.0);
    for (int i = threadIdx.x; i <= width + 1; i += blockDim.x) inv[i] = i > 0 ? 1.0 / (double)i : 0.0;
    __syncthreads();
    const long long total = bins * nperm;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long p = idx / bins, b = idx - p * bins;        // permutation-major output [P][bins][K]
        const unsigned long long gb = (unsigned long long)(bin_offset + b);
        Philox rng;
        rng.key0 = (uint32_t)seed;
        rng.key1 = (uint32_t)(seed >> 32);
        rng.ctr[0] = 0;
        rng.ctr[1] = (uint32_t)p;
        rng.ctr[2] = (uint32_t)gb;
        rng.ctr[3] = (uint32_t)(gb >> 32);
        rng.have = 0;
        int remaining = 0;
        for (int s = 0; s < K; ++s) remaining += (int)cnt_a[b * K + s] + (int)cnt_b[b * K + s];
        int need_a = min(size_a, remaining);
        int need_b = min(size_b, remaining - need_a);
        for (int s = 0; s < K; ++s) {
            const int c = (int)cnt_a[b * K + s] + (int)cnt_b[b * K + s];
            int ga = 0, gb2 = 0;
            if (c > 0) {
                ga = hypergeometric(rng, remaining, c, need_a, lf, inv);
                gb2 = hypergeometric(rng, remaining - need_a, c - ga, need_b, lf, inv);
            }
            remaining -= c;
            need_a -= ga;
            need_b -= gb2;
            out_a[idx * K + s] = (uint16_t)ga;
            out_b[idx * K + s] = (uint16_t)gb2;
        }
    }
}

// ---------------------------------------------------------------- delta / null distance
// numpy float32 pairwise summation of n < 128 contiguous values (what np.sum(axis=1) does per row):
// n < 8: left to right from 0; else 8 running sums over blocks of 8, a fixed combination tree, then the tail.
template <class F>
__device__ __forceinline__ float numpy_rowsum_f32(int n, F at) {
    if (n < 8) {
        float res = 0.f;
        for (int i = 0; i < n; ++i) res = __fadd_rn(res, at(i));
        return res;
    }
    float r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = at(k);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = __fadd_rn(r[k], at(i + k));
    }
    float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                          __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __fadd_rn(res, at(i));
    return res;
}

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
            const float sum = numpy_rowsum_f32(K, [&](int i) { return __fsub_rn(pa[i], pb[i]); });
            const float sq = numpy_rowsum_f32(K, [&](int i) {
                const float d = __fsub_rn(pa[i], pb[i]);
                return __fmul_rn(d, d);
            });
            const float sign = sum > 0.f ? 1.f : (sum < 0.f ? -1.f : (sum == 0.f ? 0.f : sum));      // np.sign (nan stays nan)
            null_dist[r] = __fmul_rn(sq, sign);
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

static unsigned grid_for(long long n, int threads, int per_sm) {
    long long blocks = (n + threads - 1) / threads;
    const long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
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

extern "C" int epi_shuffled_counts_philox(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins,
                                          int32_t K, int32_t width, int32_t size_a, int32_t size_b, uint64_t seed,
                                          int64_t bin_offset, int32_t nperm,
                                          uint16_t* cnt_a_out, uint16_t* cnt_b_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && K >= 1 && K <= EPI_MAX_STATES && nperm >= 1, "bad paired shape");
    EPI_REQUIRE(size_a >= 0 && size_b >= 0, "negative group size");
    EPI_REQUIRE(bin_offset >= 0, "negative bin offset");
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
        cnt_a_dev, cnt_b_dev, bins, K, size_a, size_b, width, (unsigned long long)seed, (long long)bin_offset, nperm, cnt_a_out,
        cnt_b_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
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
