// K5 -- S1 / S2 Kullback-Leibler scores from the per-bin uint16 counts.
//
//   S1: score[s] = o log2(o / E1[s]),            o    = c_s / width            (scores.py:339-344, 317, 550)
//   S2: score[t] = sum_s o_st log2(o_st / E2[s][t]),
//                  o_st = (c_s c_t - [s==t] c_s) / P, added in order s = 0..K-1 (scores.py:443-451, 412, 550)
//   terms with o == 0 or E == 0 are 0 (numpy.ma masking in klScoreND).
//
// Traffic per bin: 2K bytes of counts in, 4K bytes of float32 scores out (36 + 72 B at K = 18); the work is
// float64 arithmetic.  A term-by-term evaluation costs a correctly rounded divide and a log2 per (s,t) pair
// (171 distinct pairs per bin at K = 18: ~35 ms per 15.5 M bins on the fp64 pipe).  The TABLE path removes
// the transcendentals from the per-bin work:
//      log2(o_st / E_st) = L(c_s) + L(c_t) - log2 P - log2 E_st,      L = log2 of an integer count (table)
//      score[t] = (c_t / P) * { [A + W (L(c_t) - log2 P) - (LE c)_t]
//                               - c_t (2 L(c_t) - log2 P - LE_tt) + (c_t - 1)(L(c_t) + L(c_t - 1) - log2 P - LE_tt) }
//      A = sum_s c_s L(c_s),  W = sum_s c_s,  (LE c)_t = sum_s c_s log2 E_st
// i.e. one 18x18 mat-vec in DFMAs per bin.  LE lives in __constant__ memory so the DFMAs take it as a
// constant-bank operand (no load instructions); it is rebuilt from the float32 table on every call.
// The result differs from the term-by-term float64 evaluation by rounding only (tests: 1e-9 relative +
// 1e-12 absolute).  Whenever E has a zero entry (a foreign expected table) the kernel switches to the
// DIRECT evaluation, which implements the masked-term semantics literally.
//
// I/O is staged per warp (no block-wide barriers in the steady state): 32 bins of counts come in as 16-byte
// vectors, 32 rows of float32 scores leave as 16-byte vectors.
//
// Dispatch (dispatch_s2 below): with width <= 2047 the S2 TABLE evaluation runs on the tensor cores
// (tc_tables.cu: the (LE c) mat-vec as an exact int8 tcgen05 product of the count bytes with base-256 digits
// of -log2 E) and the DIRECT kernel is queued behind it, gated on the device-side "table has a zero" flag;
// wider inputs take the DFMA TABLE kernel of this file, which switches to DIRECT itself on that flag.
// S1 needs no re-association at all: its K x (width+1) value table is built with the reference expression
// itself (k5_s1_table_kernel), so S1 scores are bit-equal to the float64 reference before the float32 cast.
#include "common.cuh"

namespace epi {

constexpr int K5_THREADS = 256;
constexpr int K5_WARPS = K5_THREADS / 32;
constexpr int KT_MAX = EPI_MAX_STATES;

__constant__ __align__(16) double c_log2e[KT_MAX * KT_MAX];     // S2: log2 E[s][t], row stride KT; S1: log2 E[s]

// one CTA: expected table (float32) -> log2 table (float64, row stride kt) + zero flag, in the device workspace
__global__ void k5_prepare_kernel(const float* __restrict__ e, int rows, int cols, int kt, double* __restrict__ out,
                                  PrepFlags* flags) {
    __shared__ int zero;
    if (threadIdx.x == 0) zero = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < rows * kt; i += blockDim.x) {
        const int s = i / kt, q = i - s * kt;
        double v = 0.0;
        if (q < cols) {
            const double ev = (double)e[s * cols + q];
            if (ev > 0.0) v = log2(ev);
            else zero = 1;
        }
        out[i] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) flags->has_zero = zero;
}

__device__ __forceinline__ double kl_direct(double obs, double e) {
    // klScoreND (scores.py:550): 0 where E == 0 (masked divide) or obs/E <= 0 (masked log2)
    if (e == 0.0 || obs == 0.0) return 0.0;
    return obs * log2(obs / e);
}

// ---- per-warp staging helpers -------------------------------------------------------------------
// Per-warp stream of 32-bin count groups: two slabs filled by 1D bulk copies (cp.async.bulk + mbarrier), the
// group after the current one is always in flight while the warp computes.  The partial group at the end of
// the array is read with plain loads.
struct WarpCountStream {
    const uint16_t* cnt;
    uint16_t* slab[2];
    uint64_t* bar;        // two mbarriers
    long long bins, ngroups, stride;
    int K, lane, buf;
    uint32_t phase[2];

    __device__ __forceinline__ void issue(long long g, int b) const {
        if (lane == 0 && g < ngroups && bins - g * 32 >= 32) {
            mbar_expect_tx(&bar[b], 64 * K);
            bulk_load_1d(slab[b], cnt + g * 32 * K, 64 * K, &bar[b]);
        }
    }
    // returns the slab holding group g (its first nvalid rows); prefetches group g + stride
    __device__ __forceinline__ const uint16_t* acquire(long long g, int nvalid) {
        const int b = buf;
        buf ^= 1;
        issue(g + stride, b ^ 1);
        if (nvalid == 32) {
            mbar_wait(&bar[b], phase[b]);
            phase[b] ^= 1;
        } else {
            const uint16_t* src = cnt + g * 32 * K;
            for (int i = lane; i < nvalid * K; i += 32) slab[b][i] = src[i];
            __syncwarp();
        }
        return slab[b];
    }
};

// the warp's 32 rows of float scores -> global (16-byte stores when the group is full)
__device__ __forceinline__ void warp_store_scores(const float* slab, float* __restrict__ dst, int nvalid, int K,
                                                  int lane) {
    __syncwarp();
    if (nvalid == 32) {
        const float4* s4 = reinterpret_cast<const float4*>(slab);  // 32*K*4 bytes = 8K vectors
        float4* d4 = reinterpret_cast<float4*>(dst);
        for (int i = lane; i < 8 * K; i += 32) d4[i] = s4[i];
    } else {
        for (int i = lane; i < nvalid * K; i += 32) dst[i] = slab[i];
    }
    __syncwarp();
}

// ---- S1 -----------------------------------------------------------------------------------------
// A bin's S1 score for state s depends only on (s, c_s), and c_s <= width: all K x (width+1) possible values are
// evaluated ONCE with the reference's own formula (float64 divide, divide, log2, multiply -- scores.py:339-344, 550)
// and the per-bin work is a table look-up.  The float32 output is therefore the float32 rounding of exactly the
// float64 expression the reference evaluates (no re-association: rankings downstream, e.g. the regions of interest,
// see the same values), and the kernel is bound by its 6K bytes per bin of traffic.
constexpr int S1_SMEM_TABLE_BYTES = 96 * 1024;

__global__ void k5_s1_table_kernel(const float* __restrict__ exp1, int K, int width, float* __restrict__ v32,
                                   double* __restrict__ v64) {
    const int n = K * (width + 1);
    const double dw = (double)width;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int s = i / (width + 1), c = i - s * (width + 1);
        const double v = kl_direct((double)c / dw, (double)exp1[s]);
        v32[i] = (float)v;
        v64[i] = v;
    }
}

// THREADS: 256, or 1024 when the value table is large: the table is per CTA, so one big CTA keeps 32 warps resident on an SM
// where 256-thread CTAs with a 60 KB table each would only fit twice (16 warps; measured 0.52 ms -> see profiles/).
template <bool SMEM_TABLE, int THREADS>
__global__ void __launch_bounds__(THREADS) k5_s1_kernel(const uint16_t* __restrict__ cnt, long long bins, int K,
                                                        int width, const float* __restrict__ v32g,
                                                        const double* __restrict__ v64g,
                                                        float* __restrict__ out32, double* __restrict__ out64) {
    constexpr int K5_THREADS = THREADS, K5_WARPS = THREADS / 32;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint16_t* cslab = reinterpret_cast<uint16_t*>(smem_raw);                          // K5_WARPS * 2 * 32 * K u16
    float* fslab = reinterpret_cast<float*>(smem_raw + K5_WARPS * 32 * K * 4);        // K5_WARPS * 32 * K f32
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + K5_WARPS * 32 * K * 8);   // K5_WARPS * 2
    float* vts = reinterpret_cast<float*>(bars + K5_WARPS * 2);                       // K * (width + 1) f32

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int w1 = width + 1;
    if (tid == 0) {
        for (int i = 0; i < K5_WARPS * 2; ++i) mbar_init(&bars[i], 1);
        mbar_fence_init();
    }
    if (SMEM_TABLE)
        for (int i = tid; i < K * w1; i += K5_THREADS) vts[i] = v32g[i];
    __syncthreads();
    const float* vt = SMEM_TABLE ? vts : v32g;
    float* myf = fslab + warp * 32 * K;

    const long long ngroups = (bins + 31) / 32;
    WarpCountStream in{cnt, {cslab + warp * 64 * K, cslab + warp * 64 * K + 32 * K}, bars + warp * 2, bins, ngroups,
                       (long long)gridDim.x * K5_WARPS, K, lane, 0, {0u, 0u}};
    in.issue((long long)blockIdx.x * K5_WARPS + warp, 0);
    for (long long g = (long long)blockIdx.x * K5_WARPS + warp; g < ngroups; g += in.stride) {
        const long long bin0 = g * 32;
        const int nvalid = (int)((bins - bin0) < 32 ? (bins - bin0) : 32);
        const uint16_t* myc = in.acquire(g, nvalid);
        if (lane < nvalid) {
            const uint16_t* row = myc + lane * K;
            for (int s = 0; s < K; ++s) {
                const int c = row[s];
                myf[lane * K + s] = vt[s * w1 + c];
                if (out64 != nullptr) out64[(bin0 + lane) * K + s] = v64g[s * w1 + c];
            }
        }
        if (out32 != nullptr) warp_store_scores(myf, out32 + bin0 * K, nvalid, K, lane);
        else __syncwarp();
    }
}

// per-bin evaluation (widths beyond the table limit, and the explicit DIRECT mode)
__global__ void __launch_bounds__(K5_THREADS) k5_s1_direct_kernel(const uint16_t* __restrict__ cnt, long long bins, int K,
                                                                  int width, const float* __restrict__ exp1,
                                                                  float* __restrict__ out32, double* __restrict__ out64) {
    const double dw = (double)width;
    const long long n = bins * K;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int s = (int)(i % K);
        const double v = kl_direct((double)cnt[i] / dw, (double)__ldg(exp1 + s));
        if (out32 != nullptr) out32[i] = (float)v;
        if (out64 != nullptr) out64[i] = v;
    }
}

// ---- S2 -----------------------------------------------------------------------------------------
template <int KT>
__global__ void __launch_bounds__(K5_THREADS) k5_s2_kernel(const uint16_t* __restrict__ cnt, long long bins, int K,
                                                           int width, double perms, const float* __restrict__ exp2,
                                                           const PrepFlags* __restrict__ flags, int force_direct,
                                                           float* __restrict__ out32, double* __restrict__ out64) {
    // force_direct == 2: fallback queued behind the tensor-core kernel, runs only when the table has zero entries
    if (force_direct == 2 && !flags->has_zero) return;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint16_t* cslab = reinterpret_cast<uint16_t*>(smem_raw);                          // K5_WARPS * 2 * 32 * K u16
    float* fslab = reinterpret_cast<float*>(smem_raw + K5_WARPS * 32 * K * 4);        // K5_WARPS * 32 * K f32
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + K5_WARPS * 32 * K * 8);   // K5_WARPS * 2

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int i = 0; i < K5_WARPS * 2; ++i) mbar_init(&bars[i], 1);
        mbar_fence_init();
    }
    __syncthreads();
    const double lp = log2(perms);
    const double inv_perms = 1.0 / perms;
    const bool direct = force_direct || flags->has_zero;
    float* myf = fslab + warp * 32 * K;

    const long long ngroups = (bins + 31) / 32;
    WarpCountStream in{cnt, {cslab + warp * 64 * K, cslab + warp * 64 * K + 32 * K}, bars + warp * 2, bins, ngroups,
                       (long long)gridDim.x * K5_WARPS, K, lane, 0, {0u, 0u}};
    in.issue((long long)blockIdx.x * K5_WARPS + warp, 0);
    for (long long g = (long long)blockIdx.x * K5_WARPS + warp; g < ngroups; g += in.stride) {
        const long long bin0 = g * 32;
        const int nvalid = (int)((bins - bin0) < 32 ? (bins - bin0) : 32);
        const uint16_t* myc = in.acquire(g, nvalid);
        if (lane < nvalid) {
            const uint16_t* row = myc + lane * K;
            float* orow = myf + lane * K;
            if (direct) {
                for (int q = 0; q < K; ++q) {
                    const long long cq = row[q];
                    double sum = 0.0;
                    if (cq != 0) {
                        for (int s = 0; s < K; ++s) {
                            const long long cs = row[s];
                            const long long prod = (s == q) ? cs * (cs - 1) : cs * cq;
                            if (prod != 0) sum += kl_direct((double)prod / perms, (double)__ldg(exp2 + s * K + q));
                        }
                    }
                    orow[q] = (float)sum;
                    if (out64 != nullptr) out64[(bin0 + lane) * K + q] = sum;
                }
            } else {
                // bracket for target state t (see the header comment), after collecting terms:
                //   br = (A - (LE c)_t) + (L(c_t) - log2 P)(W - 1) - c_t L(c_t) + (c_t - 1) L(c_t - 1) + LE_tt
                double cd[KT], mc[KT];
                double a = 0.0, w = 0.0;
#pragma unroll
                for (int s = 0; s < KT; ++s) {
                    const int c = s < K ? row[s] : 0;
                    cd[s] = (double)c;
                    const double l = c > 0 ? log2((double)c) : 0.0;
                    a = fma(cd[s], l, a);
                    w += cd[s];
                    mc[s] = 0.0;
                }
                const double2* le2 = reinterpret_cast<const double2*>(c_log2e);     // KT is even: 16-byte pairs
#pragma unroll
                for (int s = 0; s < KT; ++s) {
#pragma unroll
                    for (int q = 0; q < KT; q += 2) {
                        const double2 m = le2[(s * KT + q) >> 1];
                        mc[q] = fma(cd[s], m.x, mc[q]);
                        mc[q + 1] = fma(cd[s], m.y, mc[q + 1]);
                    }
                }
                const double wm1 = w - 1.0;
#pragma unroll
                for (int q = 0; q < KT; ++q) {
                    if (q < K) {
                        const int c = row[q];
                        const int cm = c > 0 ? c - 1 : 0;
                        const double lt = c > 0 ? log2((double)c) : 0.0;
                        const double l1 = cm > 0 ? log2((double)cm) : 0.0;
                        double br = (a - mc[q]) + c_log2e[q * KT + q];
                        br = fma(lt - lp, wm1, br);
                        br = fma(-cd[q], lt, br);
                        br = fma((double)cm, l1, br);
                        const double v = c > 0 ? (cd[q] * inv_perms) * br : 0.0;   // absent state: +0.0 as in the reference
                        orow[q] = (float)v;
                        if (out64 != nullptr) out64[(bin0 + lane) * K + q] = v;
                    }
                }
            }
        }
        if (out32 != nullptr) warp_store_scores(myf, out32 + bin0 * K, nvalid, K, lane);
        else __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// builds the log2 table in the device workspace, copies it into constant memory (device-to-device, stream ordered)
static int prepare_tables(const float* e, int rows, int cols, int kt, cudaStream_t st, const PrepFlags** flags_out) {
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    k5_prepare_kernel<<<1, 256, 0, st>>>(e, rows, cols, kt, ws->log2e, &ws->prep_flags);
    EPI_CUDA(cudaGetLastError());
    EPI_CUDA(cudaMemcpyToSymbolAsync(c_log2e, ws->log2e, (size_t)rows * kt * 8, 0, cudaMemcpyDeviceToDevice, st));
    *flags_out = &ws->prep_flags;
    return 0;
}

int s1_value_table(const float* e, int K, int width, float* v32, double* v64, cudaStream_t st) {
    const int n = K * (width + 1);
    k5_s1_table_kernel<<<(n + 255) / 256, 256, 0, st>>>(e, K, width, v32, v64);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

static int launch_s1(const uint16_t* cnt, int64_t bins, int K, int width, const float* e, int direct, float* o32,
                     double* o64, cudaStream_t st) {
    if (direct || width > S1_TABLE_MAX_WIDTH) {
        int64_t blocks = (bins * K + K5_THREADS - 1) / K5_THREADS;
        const int64_t cap = (int64_t)sm_count() * 16;
        if (blocks > cap) blocks = cap;
        k5_s1_direct_kernel<<<(unsigned)blocks, K5_THREADS, 0, st>>>(cnt, bins, K, width, e, o32, o64);
        EPI_CUDA(cudaGetLastError());
        return 0;
    }
    // value table: K x (width+1) float32 + float64, in the device workspace
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    double* v64 = ws->s1_v64;
    float* v32 = ws->s1_v32;
    const int n = K * (width + 1);
    if (int rc = s1_value_table(e, K, width, v32, v64, st)) return rc;
    const size_t base = (size_t)K5_WARPS * 32 * K * 8 + K5_WARPS * 16;
    const size_t table = (size_t)n * 4;
    const int64_t ntiles = (bins + K5_THREADS - 1) / K5_THREADS;
    const size_t base_big = (size_t)32 * 32 * K * 8 + 32 * 16;          // 1024-thread CTA
    if (table <= (size_t)S1_SMEM_TABLE_BYTES && 4 * (base + table + 1024) > (size_t)220 * 1024 &&
        base_big + table + 1024 <= (size_t)226 * 1024) {
        // fewer than four 256-thread CTAs would fit next to their tables: one 1024-thread CTA per SM shares ONE table
        auto kern = k5_s1_kernel<true, 1024>;
        EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(base_big + table)));
        kern<<<persistent_grid((bins + 1023) / 1024, 1), 1024, base_big + table, st>>>(cnt, bins, K, width, v32, v64, o32, o64);
    } else if (table <= (size_t)S1_SMEM_TABLE_BYTES) {
        auto kern = k5_s1_kernel<true, K5_THREADS>;
        EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(base + table)));
        const int per_sm = (int)((size_t)220 * 1024 / (base + table + 1024));
        kern<<<persistent_grid(ntiles, per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm)), K5_THREADS, base + table, st>>>(
            cnt, bins, K, width, v32, v64, o32, o64);
    } else {
        auto kern = k5_s1_kernel<false, K5_THREADS>;
        EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)base));
        kern<<<persistent_grid(ntiles, 4), K5_THREADS, base, st>>>(cnt, bins, K, width, v32, v64, o32, o64);
    }
    EPI_CUDA(cudaGetLastError());
    return 0;
}

template <int KT>
static int launch_s2(const uint16_t* cnt, int64_t bins, int K, int width, int64_t perms, const float* e,
                     const PrepFlags* flags, int direct, float* o32, double* o64, cudaStream_t st) {
    auto kern = k5_s2_kernel<KT>;
    const size_t smem = (size_t)K5_WARPS * 32 * K * 8 + K5_WARPS * 16;
    EPI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t ntiles = (bins + K5_THREADS - 1) / K5_THREADS;
    kern<<<persistent_grid(ntiles, 3), K5_THREADS, smem, st>>>(cnt, bins, K, width, (double)perms, e, flags, direct, o32,
                                                                o64);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

template <int KT>
static int dispatch_s2(const uint16_t* cnt, int64_t bins, int K, int width, int64_t perms, const float* e, float* o32,
                       double* o64, int mode, cudaStream_t st) {
    const PrepFlags* flags = nullptr;
    if (mode == EPI_SCORE_TABLE && scores_s2_tc_eligible(width)) {
        // tensor-core mat-vec (tc_tables.cu); a table with zero entries makes it a no-op and un-gates the DIRECT kernel
        DeviceWorkspace* ws = device_workspace();
        EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
        PrepFlags* fl = &ws->prep_flags;
        if (int rc = scores_s2_tc(cnt, bins, K, width, perms, e, &fl->has_zero, o32, o64, st)) return rc;
        return launch_s2<KT>(cnt, bins, K, width, perms, e, fl, 2, o32, o64, st);
    }
    if (int rc = prepare_tables(e, K, K, KT, st, &flags)) return rc;
    return launch_s2<KT>(cnt, bins, K, width, perms, e, flags, mode == EPI_SCORE_DIRECT, o32, o64, st);
}

}  // namespace epi

using namespace epi;

static int check_score_args(const void* cnt, int64_t bins, int K, int width, const void* e, int mode) {
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && bins < (1ll << 31), "bins=%lld out of range", (long long)bins);
    EPI_REQUIRE(K >= 1 && K <= EPI_MAX_STATES, "num_states=%d out of range [1, %d]", K, EPI_MAX_STATES);
    EPI_REQUIRE(width >= 1 && width <= 65535, "width=%d out of range [1, 65535]", width);
    EPI_REQUIRE(mode == EPI_SCORE_TABLE || mode == EPI_SCORE_DIRECT, "unknown score mode %d", mode);
    if (bins == 0) return 0;
    EPI_REQUIRE(cnt != nullptr && e != nullptr, "null pointer argument");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(cnt) & 15) == 0, "cnt_dev must be 16-byte aligned");
    return 0;
}

extern "C" int epi_scores_s1(const uint16_t* cnt_dev, int64_t bins, int32_t K, int32_t width, const float* exp1_dev,
                             float* out32_dev, double* out64_dev, int32_t mode, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_score_args(cnt_dev, bins, K, width, exp1_dev, mode)) return rc;
    if (bins == 0 || (out32_dev == nullptr && out64_dev == nullptr)) return 0;
    EPI_REQUIRE(out32_dev == nullptr || (reinterpret_cast<uintptr_t>(out32_dev) & 15) == 0,
                "out32_dev must be 16-byte aligned");
    return launch_s1(cnt_dev, bins, K, width, exp1_dev, mode == EPI_SCORE_DIRECT, out32_dev, out64_dev, st);
}

extern "C" int epi_scores_s2_fixed_point(const float* exp2_dev, int32_t K, int64_t perms, uint64_t* mfix_dev,
                                         int32_t* fraction_bits_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(K >= 1 && K <= EPI_MAX_STATES, "num_states=%d out of range [1, %d]", K, EPI_MAX_STATES);
    EPI_REQUIRE(perms >= 1 && exp2_dev != nullptr && mfix_dev != nullptr, "bad argument");
    int fbits = 0;
    if (int rc = scores_s2_tc_fixed_point(exp2_dev, K, perms, reinterpret_cast<unsigned long long*>(mfix_dev), &fbits, st))
        return rc;
    if (fraction_bits_out) *fraction_bits_out = fbits;
    return 0;
}

extern "C" int epi_scores_s2(const uint16_t* cnt_dev, int64_t bins, int32_t K, int32_t width, int64_t perms,
                             const float* exp2_dev, float* out32_dev, double* out64_dev, int32_t mode, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_score_args(cnt_dev, bins, K, width, exp2_dev, mode)) return rc;
    EPI_REQUIRE(perms >= 1, "perms=%lld must be positive (needs at least 2 biosamples)", (long long)perms);
    if (bins == 0 || (out32_dev == nullptr && out64_dev == nullptr)) return 0;
    EPI_REQUIRE(out32_dev == nullptr || (reinterpret_cast<uintptr_t>(out32_dev) & 15) == 0,
                "out32_dev must be 16-byte aligned");
    if (K <= 16) return dispatch_s2<16>(cnt_dev, bins, K, width, perms, exp2_dev, out32_dev, out64_dev, mode, st);
    if (K <= 18) return dispatch_s2<18>(cnt_dev, bins, K, width, perms, exp2_dev, out32_dev, out64_dev, mode, st);
    return dispatch_s2<32>(cnt_dev, bins, K, width, perms, exp2_dev, out32_dev, out64_dev, mode, st);
}
