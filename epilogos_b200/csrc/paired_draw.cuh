// Pieces shared by the paired-mode and multi-group kernels: the shuffle samplers of epi_shuffled_counts_philox
// (pairwise.cu) and epi_multigroup_shuffled_counts_range (multigroup.cu), numpy's float32 row summation of
// epi_pairwise_combine, the multi-group statistic, and the thread groups and launch of the fused permutation kernels.
// The fused kernels (permutations.cu, multigroup.cu) draw and reduce with these same functions, so their counts are the
// composed paths' bit for bit.
#pragma once
#include "common.cuh"

namespace epi {

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

// The Philox stream of one shuffle, keyed by (seed; permutation p, GLOBAL bin index gb).
__device__ __forceinline__ Philox shuffle_stream(unsigned long long seed, uint32_t p, unsigned long long gb) {
    Philox rng;
    rng.key0 = (uint32_t)seed;
    rng.key1 = (uint32_t)(seed >> 32);
    rng.ctr[0] = 0;
    rng.ctr[1] = p;
    rng.ctr[2] = (uint32_t)gb;
    rng.ctr[3] = (uint32_t)(gb >> 32);
    rng.have = 0;
    return rng;
}

// One uniform shuffle of a bin's combined row split into A' (size_a labels) and B' (size_b labels).  For count-based
// scores it is a multivariate hypergeometric draw: walking over the states,
//   a'_s ~ HG(remaining labels, c_s, still needed by A'),  b'_s ~ HG(remaining - needed by A', c_s - a'_s, needed by B').
// emit(s, a'_s, b'_s) is called for s = 0..K-1 in order.  draw_multigroup_shuffle at G = 2 with sizes {size_a, size_b}
// and the combined row draws the same counts from the same Philox words (tests/test_multigroup_gpu.py checks it), but
// with it the fused permutation kernel ran 1.0 % slower and the composed path 0.06 % slower on an NVIDIA B200 at 1000 W,
// beyond the spread of alternated runs (profiles/r08_paired_draw_g2.jsonl), so the paired kernels keep this form.
template <class Emit>
__device__ __forceinline__ void draw_shuffle(Philox& rng, const uint16_t* __restrict__ ca, const uint16_t* __restrict__ cb,
                                             int K, int size_a, int size_b, const double* __restrict__ lf,
                                             const double* __restrict__ inv, Emit emit) {
    int remaining = 0;
    for (int s = 0; s < K; ++s) remaining += (int)ca[s] + (int)cb[s];
    int need_a = min(size_a, remaining);
    int need_b = min(size_b, remaining - need_a);
    for (int s = 0; s < K; ++s) {
        const int c = (int)ca[s] + (int)cb[s];
        int ga = 0, gb2 = 0;
        if (c > 0) {
            ga = hypergeometric(rng, remaining, c, need_a, lf, inv);
            gb2 = hypergeometric(rng, remaining - need_a, c - ga, need_b, lf, inv);
        }
        remaining -= c;
        need_a -= ga;
        need_b -= gb2;
        emit(s, ga, gb2);
    }
}

// One uniform shuffle of a bin's labels over G groups (multigroup.cu): a multivariate hypergeometric draw.  comb(s) is
// the bin's count of state s over the row being shuffled, size[g] the labels group g receives, and need(g) a per-thread
// int slot the draw keeps group g's still-needed count in.  For every state s in order and every group g in order,
//   x_gs ~ HG(labels still unassigned, labels of state s still unassigned, labels group g still needs);
// emit(s, g, x_gs) is called in that order and end_state(s) after the last group of a state.  When the sizes sum to
// less than the row (-g), the labels no group takes are left out.  When they cover the row, the last group's draw is
// deterministic and consumes no Philox word.
template <class Comb, class Need, class Emit, class EndState>
__device__ __forceinline__ void draw_multigroup_shuffle(Philox& rng, int K, int G, const int* size, Comb comb, Need need,
                                                        const double* __restrict__ lf, const double* __restrict__ inv,
                                                        Emit emit, EndState end_state) {
    int remaining = 0;
    for (int s = 0; s < K; ++s) remaining += comb(s);
    int left = remaining;
    for (int g = 0; g < G; ++g) {
        const int n = min(size[g], left);
        need(g) = n;
        left -= n;
    }
    for (int s = 0; s < K; ++s) {
        const int c = comb(s);
        int pop = remaining, succ = c;
        for (int g = 0; g < G; ++g) {
            const int ng = need(g);
            const int x = succ > 0 ? hypergeometric(rng, pop, succ, ng, lf, inv) : 0;
            pop -= ng;
            succ -= x;
            need(g) = ng - x;
            emit(s, g, x);
        }
        remaining -= c;
        end_state(s);
    }
}

// The multi-group statistic, one state at a time, in float64 without contraction (the numpy oracle computes the same
// numbers): m[s] = (sum_g n_g S_g[s]) / N, then t += n_g (S_g[s] - m[s])^2 for g in order, in one running sum over s
// outer, g inner; T = t / N.  score(g) = S_g[s] of the state at hand.
template <class F>
__device__ __forceinline__ double multigroup_mean(int G, const int* n, double N, F score) {
    double m = 0.0;
    for (int g = 0; g < G; ++g) m = __dadd_rn(m, __dmul_rn((double)n[g], (double)score(g)));
    return __ddiv_rn(m, N);
}

template <class F>
__device__ __forceinline__ double multigroup_add_state(double t, int G, const int* n, double m, F score) {
    for (int g = 0; g < G; ++g) {
        const double d = __dsub_rn((double)score(g), m);
        t = __dadd_rn(t, __dmul_rn((double)n[g], __dmul_rn(d, d)));
    }
    return t;
}

// shared-memory tables of the sampler: log(i!), i = 0..width, then 1/i, i = 0..width+1
__device__ __forceinline__ void fill_draw_tables(double* lf, double* inv, int width) {
    for (int i = threadIdx.x; i <= width; i += blockDim.x) lf[i] = lgamma((double)i + 1.0);
    for (int i = threadIdx.x; i <= width + 1; i += blockDim.x) inv[i] = i > 0 ? 1.0 / (double)i : 0.0;
}

// The fused permutation kernels give each bin to a group of T threads (T divides 32: a group never straddles a warp);
// thread t of the group takes permutations t, t + T, ...  group_mask is the calling thread's group, group_sum the sum of
// c over it.
template <int T>
__device__ __forceinline__ unsigned group_mask() {
    const int lane = threadIdx.x & 31;
    return T == 32 ? 0xffffffffu : (((1u << (T % 32)) - 1u) << (lane & ~(T - 1)));
}

template <int T>
__device__ __forceinline__ uint32_t group_sum(unsigned gmask, uint32_t c) {
#pragma unroll
    for (int off = T / 2; off > 0; off >>= 1) c += __shfl_xor_sync(gmask, c, off);
    return c;
}

// Every entry point that draws permutations perm_offset .. perm_offset + nperm - 1 of the bins from bin_offset on: the
// permutation word of the stream key (shuffle_stream) is 32 bits wide.
static inline int check_perm_range(int64_t bin_offset, int64_t perm_offset, int32_t nperm) {
    EPI_REQUIRE(bin_offset >= 0, "negative bin offset");
    EPI_REQUIRE(nperm >= 0 && perm_offset >= 0 && perm_offset + nperm <= (1ll << 32),
                "permutations %lld..%lld outside the 32-bit stream key", (long long)perm_offset,
                (long long)perm_offset + nperm - 1);
    return 0;
}

// Launches a fused permutation kernel with T = 32 / 8 / 1 threads per bin (k32, k8, k1) for nperm >= 32 / >= 8 / fewer,
// in CTAs of `threads` threads with smem(T) bytes of dynamic shared memory, on no more CTAs than stay resident at once.
template <class... P, class Smem, class... A>
static int launch_fused(void (*k32)(P...), void (*k8)(P...), void (*k1)(P...), int nperm, long long bins, int threads,
                        Smem smem, cudaStream_t st, A... args) {
    const int T = nperm >= 32 ? 32 : (nperm >= 8 ? 8 : 1);
    auto kern = T == 32 ? k32 : (T == 8 ? k8 : k1);
    const size_t bytes = smem(T);
    EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    int per_sm = 0;
    EPI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, bytes));
    kern<<<grid_for(bins, threads / T, per_sm < 1 ? 1 : per_sm), threads, bytes, st>>>(args...);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

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

// sum_s d_s^2 * sign(sum_s d_s), float32 in numpy's order, of d_s = at(s) (scores.py:231-232)
template <class F>
__device__ __forceinline__ float signed_sq_distance(int K, F at) {
    const float sum = numpy_rowsum_f32(K, at);
    const float sq = numpy_rowsum_f32(K, [&](int i) {
        const float d = at(i);
        return __fmul_rn(d, d);
    });
    const float sign = sum > 0.f ? 1.f : (sum < 0.f ? -1.f : (sum == 0.f ? 0.f : sum));      // np.sign (nan stays nan)
    return __fmul_rn(sq, sign);
}

}  // namespace epi
