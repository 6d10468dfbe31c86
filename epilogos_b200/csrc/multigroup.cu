// K10 -- multi-group comparisons: one per-bin test of whether G >= 2 disjoint groups of biosamples differ, with
// permutation counts drawn and counted on the device.
//
// Group g (n_g biosamples, N = sum_g n_g) has the score vector S_g = score of its counts at width n_g against the
// background of the union of the groups.  Per bin, in float64 without contraction (paired_draw.cuh):
//   m[s] = (sum_g n_g S_g[s]) / N,   T = (sum_s sum_g n_g (S_g[s] - m[s])^2) / N       (s outer, g inner, one running sum)
// the size-weighted between-group sum of squares; and its driver
//   g* = argmax_g n_g sum_s (S_g[s] - m[s])^2,  s* = argmax_s |S_g*[s] - m[s]|,  sign(S_g*[s*] - m[s*])   (first on ties).
// Shuffle p of bin b is draw_multigroup_shuffle with the stream shuffle_stream(seed, p, global bin); the count is
//   k[b] += #{ p : T_null(b, p) >= T[b] }.
//
//   epi_multigroup_stat                   G score arrays in; T, g*, s* and the sign out, one thread per bin.
//   epi_multigroup_shuffled_counts_range  the G-way sampler: [nperm][G][bins][K] counts of permutations from an offset on.
//   epi_multigroup_null_exceedances       the counting step of the composed path: [nperm][G][bins][K] scores in.
//   epi_multigroup_exceedances_s1         the fused S1 path: per (bin, permutation) it draws, looks S_g up in G K5-S1
//                                         value tables (s1_value_table at width n_g), forms T_null and compares.  Nothing
//                                         per (bin, permutation) goes to memory; bit-equal to the composed path.
#include "paired_draw.cuh"

namespace epi {

struct GroupSizes {
    int n[EPI_MAX_GROUPS];
};

constexpr int K10_THREADS = 256;
constexpr int K10_STAT_THREADS = 128;

// m[s] lives in shared memory, m[s * blockDim + thread]: the driver needs it after T is complete.
__global__ void __launch_bounds__(K10_STAT_THREADS) multigroup_stat_kernel(const float* __restrict__ sc, int G,
                                                                           long long bins, int K, GroupSizes sz, int N,
                                                                           double* __restrict__ t_out,
                                                                           uint8_t* __restrict__ g_out,
                                                                           uint8_t* __restrict__ s_out,
                                                                           int8_t* __restrict__ sign_out) {
    extern __shared__ double msh[];
    double* m = msh + threadIdx.x;
    const long long gs = bins * K;
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < bins;
         b += (long long)gridDim.x * blockDim.x) {
        const float* p = sc + b * K;
        double t = 0.0;
        for (int s = 0; s < K; ++s) {
            auto score = [&](int g) { return p[g * gs + s]; };
            const double ms = multigroup_mean(G, sz.n, (double)N, score);
            m[s * K10_STAT_THREADS] = ms;
            t = multigroup_add_state(t, G, sz.n, ms, score);
        }
        int gbest = 0;
        double vbest = -1.0;
        for (int g = 0; g < G; ++g) {
            double acc = 0.0;
            for (int s = 0; s < K; ++s) {
                const double d = __dsub_rn((double)p[g * gs + s], m[s * K10_STAT_THREADS]);
                acc = __dadd_rn(acc, __dmul_rn(d, d));
            }
            const double v = __dmul_rn((double)sz.n[g], acc);
            if (v > vbest) {
                vbest = v;
                gbest = g;
            }
        }
        int sbest = 0;
        double dbest = -1.0, dsel = 0.0;
        for (int s = 0; s < K; ++s) {
            const double d = __dsub_rn((double)p[gbest * gs + s], m[s * K10_STAT_THREADS]);
            if (fabs(d) > dbest) {
                dbest = fabs(d);
                dsel = d;
                sbest = s;
            }
        }
        t_out[b] = __ddiv_rn(t, (double)N);
        g_out[b] = (uint8_t)gbest;
        s_out[b] = (uint8_t)sbest;
        sign_out[b] = dsel < 0.0 ? -1 : 1;
    }
}

// One thread per (bin, permutation).  Shared memory: the sampler's tables (2 N + 3 doubles), then each thread's
// still-needed counts, need[g * blockDim + thread].
__global__ void __launch_bounds__(K10_THREADS) multigroup_shuffled_counts_kernel(
    const uint16_t* __restrict__ cnt, long long gstride, int G, long long bins, int K, GroupSizes sz, int N,
    unsigned long long seed, long long bin_offset, long long perm_offset, int nperm, uint16_t* __restrict__ out) {
    extern __shared__ double lf[];
    double* inv = lf + (N + 1);
    int* need = reinterpret_cast<int*>(inv + (N + 2)) + threadIdx.x;
    fill_draw_tables(lf, inv, N);
    __syncthreads();
    const long long total = bins * nperm;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long p = idx / bins, b = idx - p * bins;
        Philox rng = shuffle_stream(seed, (uint32_t)(perm_offset + p), (unsigned long long)(bin_offset + b));
        const uint16_t* c = cnt + b * K;
        uint16_t* o = out + (p * G * bins + b) * K;
        draw_multigroup_shuffle(
            rng, K, G, sz.n,
            [&](int s) {
                int v = 0;
                for (int g = 0; g < G; ++g) v += (int)c[g * gstride + s];
                return v;
            },
            [&](int g) -> int& { return need[g * K10_THREADS]; }, lf, inv,
            [&](int s, int g, int x) { o[(long long)g * bins * K + s] = (uint16_t)x; }, [](int) {});
    }
}

// One thread per bin; it walks the permutations of its bin.
__global__ void __launch_bounds__(K10_THREADS) multigroup_null_exceedances_kernel(
    const float* __restrict__ sc, int G, int nperm, long long bins, int K, GroupSizes sz, int N,
    const double* __restrict__ tb, uint32_t* __restrict__ k) {
    const long long gs = bins * K;
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < bins;
         b += (long long)gridDim.x * blockDim.x) {
        const double thr = tb[b];
        uint32_t c = 0;
        for (int p = 0; p < nperm; ++p) {
            const float* q = sc + (long long)p * G * gs + b * K;
            double t = 0.0;
            for (int s = 0; s < K; ++s) {
                auto score = [&](int g) { return q[g * gs + s]; };
                t = multigroup_add_state(t, G, sz.n, multigroup_mean(G, sz.n, (double)N, score), score);
            }
            c += __ddiv_rn(t, (double)N) >= thr ? 1u : 0u;
        }
        k[b] += c;
    }
}

// T threads own one bin (T divides 32); thread t takes permutations t, t + T, ...  Shared memory, in order:
//   the sampler's tables                    (2 N + 3) doubles
//   the G value tables, group g at voff[g]  K (n_g + 1) floats each
//   per thread, still-needed counts         uint16 [G][K10_THREADS]
//   per thread, the current state's draws   uint16 [G][K10_THREADS]
//   per bin slot, the union's counts        uint16 [K10_THREADS / T][K]
struct ValueOffsets {
    int off[EPI_MAX_GROUPS];
};

template <int T>
__global__ void __launch_bounds__(K10_THREADS) multigroup_exceedances_s1_kernel(
    const uint16_t* __restrict__ cnt, long long gstride, int G, long long bins, int K, GroupSizes sz, int N,
    unsigned long long seed, long long bin_offset, long long perm_offset, int nperm, const float* __restrict__ vt_g,
    ValueOffsets vo, int nvt, const double* __restrict__ tb, uint32_t* __restrict__ k) {
    extern __shared__ double lf[];
    double* inv = lf + (N + 1);
    float* vt = reinterpret_cast<float*>(inv + (N + 2));
    uint16_t* need = reinterpret_cast<uint16_t*>(vt + nvt) + threadIdx.x;
    uint16_t* drawn = need + G * K10_THREADS;
    constexpr int SLOTS = K10_THREADS / T;
    uint16_t* comb_all = need - threadIdx.x + 2 * G * K10_THREADS;
    fill_draw_tables(lf, inv, N);
    for (int i = threadIdx.x; i < nvt; i += blockDim.x) vt[i] = vt_g[i];
    __syncthreads();
    uint16_t* comb = comb_all + (threadIdx.x / T) * K;
    const int t = threadIdx.x % T;
    const unsigned gmask = group_mask<T>();
    const double dN = (double)N;
    for (long long b = blockIdx.x * (long long)SLOTS + threadIdx.x / T; b < bins; b += (long long)gridDim.x * SLOTS) {
        const double thr = tb[b];
        __syncwarp(gmask);                                   // the previous bin's readers are done with comb
        for (int s = t; s < K; s += T) {
            int v = 0;
            for (int g = 0; g < G; ++g) v += (int)cnt[g * gstride + b * K + s];
            comb[s] = (uint16_t)v;
        }
        __syncwarp(gmask);
        const unsigned long long gb = (unsigned long long)(bin_offset + b);
        uint32_t c = 0;
        for (int p = t; p < nperm; p += T) {
            Philox rng = shuffle_stream(seed, (uint32_t)(perm_offset + p), gb);
            double tn = 0.0, msum = 0.0;
            int cur = 0;
            auto score = [&](int g) { return vt[vo.off[g] + cur * (sz.n[g] + 1) + (int)drawn[g * K10_THREADS]]; };
            draw_multigroup_shuffle(
                rng, K, G, sz.n, [&](int s) { return (int)comb[s]; },
                [&](int g) -> uint16_t& { return need[g * K10_THREADS]; }, lf, inv,
                [&](int s, int g, int x) {
                    drawn[g * K10_THREADS] = (uint16_t)x;
                    msum = __dadd_rn(msum, __dmul_rn((double)sz.n[g], (double)vt[vo.off[g] + s * (sz.n[g] + 1) + x]));
                },
                [&](int s) {
                    cur = s;
                    tn = multigroup_add_state(tn, G, sz.n, __ddiv_rn(msum, dN), score);
                    msum = 0.0;
                });
            c += __ddiv_rn(tn, dN) >= thr ? 1u : 0u;
        }
        c = group_sum<T>(gmask, c);
        if (t == 0) k[b] += c;
    }
}

}  // namespace epi

using namespace epi;

// checks the group list and fills the kernel's copy; returns 0 or an error code with the message set
static int read_sizes(const int32_t* sizes, int G, GroupSizes* sz, int* N) {
    EPI_REQUIRE(G >= 2 && G <= EPI_MAX_GROUPS, "groups=%d out of range [2, %d]", G, EPI_MAX_GROUPS);
    EPI_REQUIRE(sizes != nullptr, "null pointer argument");
    long long total = 0;
    for (int g = 0; g < G; ++g) {
        EPI_REQUIRE(sizes[g] >= 1, "group %d has %d biosamples", g, sizes[g]);
        sz->n[g] = sizes[g];
        total += sizes[g];
    }
    for (int g = G; g < EPI_MAX_GROUPS; ++g) sz->n[g] = 0;
    EPI_REQUIRE(total <= 65535, "%lld biosamples in the groups, more than 65535", total);
    *N = (int)total;
    return 0;
}

extern "C" int epi_multigroup_stat(const float* scores_dev, int32_t groups, int64_t bins, int32_t num_states,
                                   const int32_t* sizes, double* t_out, uint8_t* group_out, uint8_t* state_out,
                                   int8_t* sign_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && num_states >= 1 && num_states <= EPI_MAX_STATES, "bad multi-group shape");
    GroupSizes sz;
    int N = 0;
    if (int rc = read_sizes(sizes, groups, &sz, &N)) return rc;
    if (bins == 0) return 0;
    EPI_REQUIRE(scores_dev && t_out && group_out && state_out && sign_out, "null pointer argument");
    const size_t smem = (size_t)num_states * K10_STAT_THREADS * 8;
    EPI_CUDA(cudaFuncSetAttribute(multigroup_stat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    multigroup_stat_kernel<<<grid_for(bins, K10_STAT_THREADS, 8), K10_STAT_THREADS, smem, st>>>(
        scores_dev, groups, bins, num_states, sz, N, t_out, group_out, state_out, sign_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_multigroup_shuffled_counts_range(const uint16_t* cnt_dev, int64_t group_stride, int32_t groups,
                                                    int64_t bins, int32_t num_states, const int32_t* sizes,
                                                    uint64_t seed, int64_t bin_offset, int64_t perm_offset,
                                                    int32_t nperm, uint16_t* out_dev, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && num_states >= 1 && num_states <= EPI_MAX_STATES, "bad multi-group shape");
    EPI_REQUIRE(group_stride >= bins * num_states, "group stride %lld shorter than a group's %lld counts",
                (long long)group_stride, (long long)(bins * num_states));
    GroupSizes sz;
    int N = 0;
    if (int rc = read_sizes(sizes, groups, &sz, &N)) return rc;
    if (int rc = check_perm_range(bin_offset, perm_offset, nperm)) return rc;
    if (bins == 0 || nperm == 0) return 0;
    EPI_REQUIRE(cnt_dev && out_dev, "null pointer argument");
    const size_t smem = (size_t)(2 * N + 3) * 8 + (size_t)groups * K10_THREADS * 4;
    EPI_REQUIRE(smem <= 200 * 1024, "too many biosamples (%d in %d groups) for the shuffle kernel", N, groups);
    EPI_CUDA(cudaFuncSetAttribute(multigroup_shuffled_counts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
    int per_sm = 0;
    EPI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, multigroup_shuffled_counts_kernel, K10_THREADS, smem));
    multigroup_shuffled_counts_kernel<<<grid_for(bins * nperm, K10_THREADS, per_sm < 1 ? 1 : per_sm), K10_THREADS, smem,
                                        st>>>(cnt_dev, (long long)group_stride, groups, bins, num_states, sz, N,
                                              (unsigned long long)seed, (long long)bin_offset, (long long)perm_offset,
                                              nperm, out_dev);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_multigroup_null_exceedances(const float* null_dev, int32_t groups, int32_t nperm, int64_t bins,
                                               int32_t num_states, const int32_t* sizes, const double* t_dev,
                                               uint32_t* k_inout, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && nperm >= 0 && num_states >= 1 && num_states <= EPI_MAX_STATES, "bad multi-group shape");
    GroupSizes sz;
    int N = 0;
    if (int rc = read_sizes(sizes, groups, &sz, &N)) return rc;
    if (bins == 0 || nperm == 0) return 0;
    EPI_REQUIRE(null_dev && t_dev && k_inout, "null pointer argument");
    multigroup_null_exceedances_kernel<<<grid_for(bins, K10_THREADS, 8), K10_THREADS, 0, st>>>(
        null_dev, groups, nperm, bins, num_states, sz, N, t_dev, k_inout);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

// shared memory of the fused kernel with T threads per bin
static size_t mg_fused_smem(int G, int K, int N, int nvt, int T) {
    return (size_t)(2 * N + 3) * 8 + (size_t)nvt * 4 + (size_t)G * K10_THREADS * 4 + (size_t)(K10_THREADS / T) * K * 2;
}

extern "C" int epi_multigroup_s1_fused_fits(int32_t groups, int32_t num_states, const int32_t* sizes) {
    if (groups < 2 || groups > EPI_MAX_GROUPS || num_states < 1 || num_states > EPI_MAX_STATES || sizes == nullptr)
        return 0;
    int n = 0, nvt = 0;
    for (int g = 0; g < groups; ++g) {
        if (sizes[g] < 1 || sizes[g] > S1_TABLE_MAX_WIDTH) return 0;
        n += sizes[g];
        nvt += num_states * (sizes[g] + 1);
    }
    // checked for one thread per bin, the launch with the most bin slots
    return n <= 65535 && mg_fused_smem(groups, num_states, n, nvt, 1) <= 200 * 1024 ? 1 : 0;
}

extern "C" int epi_multigroup_exceedances_s1(const uint16_t* cnt_dev, int64_t group_stride, int32_t groups,
                                             int64_t bins, int32_t num_states, const int32_t* sizes, uint64_t seed,
                                             int64_t bin_offset, int64_t perm_offset, int32_t nperm,
                                             const float* exp1_dev, const double* t_dev, uint32_t* k_inout,
                                             void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    const int K = num_states;
    EPI_REQUIRE(bins >= 0 && K >= 1 && K <= EPI_MAX_STATES, "bad multi-group shape");
    EPI_REQUIRE(group_stride >= bins * K, "group stride %lld shorter than a group's %lld counts",
                (long long)group_stride, (long long)(bins * K));
    GroupSizes sz;
    int N = 0;
    if (int rc = read_sizes(sizes, groups, &sz, &N)) return rc;
    if (int rc = check_perm_range(bin_offset, perm_offset, nperm)) return rc;
    ValueOffsets vo;
    int nvt = 0;
    for (int g = 0; g < groups; ++g) {
        EPI_REQUIRE(sz.n[g] <= S1_TABLE_MAX_WIDTH, "group %d has %d biosamples, more than the S1 value table's %d", g,
                    sz.n[g], S1_TABLE_MAX_WIDTH);
        vo.off[g] = nvt;
        nvt += K * (sz.n[g] + 1);
    }
    EPI_REQUIRE(epi_multigroup_s1_fused_fits(groups, K, sizes),
                "the value tables of %d groups (%d biosamples, %d states) exceed shared memory", groups, N, K);
    if (bins == 0 || nperm == 0) return 0;
    EPI_REQUIRE(cnt_dev && exp1_dev && t_dev && k_inout, "null pointer argument");
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    // the G tables side by side in the two permutation tables' space (nvt * 4 < 200 KB, far below it); the float64 halves
    // all go to the S1 scratch table and are not read
    static_assert(sizeof(ws->perm_v32) >= 200 * 1024, "the multi-group value tables share the permutation tables' space");
    float* vt = &ws->perm_v32[0][0];
    for (int g = 0; g < groups; ++g)
        if (int rc = s1_value_table(exp1_dev, K, sz.n[g], vt + vo.off[g], ws->s1_v64, st)) return rc;
    return launch_fused(multigroup_exceedances_s1_kernel<32>, multigroup_exceedances_s1_kernel<8>,
                        multigroup_exceedances_s1_kernel<1>, nperm, bins, K10_THREADS,
                        [&](int T) { return mg_fused_smem(groups, K, N, nvt, T); }, st, cnt_dev, (long long)group_stride,
                        groups, bins, K, sz, N, (unsigned long long)seed, (long long)bin_offset, (long long)perm_offset,
                        nperm, vt, vo, nvt, t_dev, k_inout);
}
