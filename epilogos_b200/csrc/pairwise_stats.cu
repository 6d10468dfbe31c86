// Paired statistics stage (step 4 of paired mode, roiAndVisualPairwise.py:177-242): the null pool, its subsamples, the
// generalized-normal fits, per-bin p-values and the Benjamini-Hochberg adjustment.
//
//   epi_null_compact      non-quiescent null distances of every permutation, in stable order (block scan + scatter)
//   epi_null_subsample    trial t takes the first S images of a keyed pseudo-random permutation of [0, N): a cycle-walking
//                         Feistel network whose round function is Philox4x32-10 keyed by (seed, t); indices and samples out
//   epi_gennorm_fit       one CTA per trial runs scipy's rv_continuous.fit for gennorm: optimize.fmin (Nelder-Mead, the
//                         control flow of _minimize_neldermead) on _penalized_nnlf from _fitstart.  Every thread of the
//                         CTA runs the same simplex logic on identical values; an objective evaluation is a fixed-order
//                         block reduction, so the fit is bit-reproducible run to run
//   epi_gennorm_pvalues   p = Q(1/beta, (|x - loc| / scale)^beta), the regularized upper incomplete gamma
//   epi_bh_adjust         LSD radix sort of the p-value bits with an index payload, reverse cumulative minimum of
//                         p_sorted / (rank / n), clip at 1, scatter back (statsmodels multipletests fdr_bh)
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace epi {

static unsigned grid_for_n(long long n, int threads, int per_sm) {
    long long blocks = (n + threads - 1) / threads;
    const long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
}

static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// ---------------------------------------------------------------- block scans (blockDim.x a multiple of 32, <= 1024)
// Exclusive prefix sum of one value per thread; *total receives the block sum.  `sh` holds 32 entries.
template <typename T>
__device__ __forceinline__ T block_exclusive_sum(T v, T* sh, T* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sh[warp] = x;
    __syncthreads();
    if (warp == 0) {
        T w = lane < nw ? sh[lane] : T(0);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        sh[lane] = w;                               // inclusive warp totals
    }
    __syncthreads();
    const T before = (warp ? sh[warp - 1] : T(0)) + x - v;
    *total = sh[nw - 1];
    __syncthreads();
    return before;
}

// Minimum over the threads AFTER this one (exclusive suffix minimum, +inf for the last thread).  `sh` holds 32 entries.
__device__ __forceinline__ double block_exclusive_suffix_min(double v, double* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    double x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_down_sync(0xffffffffu, x, o);
        if (lane + o < 32) x = fmin(x, y);
    }
    if (lane == 0) sh[warp] = x;                    // minimum of the warp
    __syncthreads();
    if (warp == 0) {
        double w = lane < nw ? sh[lane] : INFINITY;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_down_sync(0xffffffffu, w, o);
            if (lane + o < 32) w = fmin(w, y);
        }
        sh[lane] = w;                               // inclusive suffix minimum over the warps
    }
    __syncthreads();
    double after = __shfl_down_sync(0xffffffffu, x, 1);
    if (lane == 31) after = INFINITY;
    if (warp + 1 < nw) after = fmin(after, sh[warp + 1]);
    __syncthreads();
    return after;
}

// ---------------------------------------------------------------- null compaction
constexpr int NC_THREADS = 256, NC_ITEMS = 8, NC_TILE = NC_THREADS * NC_ITEMS;

__device__ __forceinline__ int nc_thread_count(const uint8_t* __restrict__ q, long long bins, long long first) {
    int c = 0;
#pragma unroll
    for (int i = 0; i < NC_ITEMS; ++i) c += (first + i < bins && (q == nullptr || q[first + i] == 0)) ? 1 : 0;
    return c;
}

__global__ void __launch_bounds__(NC_THREADS) null_compact_count_kernel(const uint8_t* __restrict__ q, long long bins,
                                                                        long long* __restrict__ blk) {
    __shared__ long long sh[32];
    const long long first = (long long)blockIdx.x * NC_TILE + (long long)threadIdx.x * NC_ITEMS;
    long long total;
    block_exclusive_sum<long long>(nc_thread_count(q, bins, first), sh, &total);
    if (threadIdx.x == 0) blk[blockIdx.x] = total;
}

// one block of 1024 threads: exclusive scan of the per-tile counts in place, grand total to *total
__global__ void __launch_bounds__(1024) exclusive_scan_ll_kernel(long long* __restrict__ v, long long n,
                                                                 long long* __restrict__ total) {
    __shared__ long long sh[32];
    const long long per = (n + blockDim.x - 1) / blockDim.x;
    const long long lo = min(n, per * threadIdx.x), hi = min(n, lo + per);
    long long s = 0;
    for (long long i = lo; i < hi; ++i) s += v[i];
    long long all;
    long long run = block_exclusive_sum<long long>(s, sh, &all);
    for (long long i = lo; i < hi; ++i) {
        const long long c = v[i];
        v[i] = run;
        run += c;
    }
    if (threadIdx.x == 0) *total = all;
}

__global__ void __launch_bounds__(NC_THREADS) null_compact_scatter_kernel(const float* __restrict__ null_dist,
                                                                          const uint8_t* __restrict__ q, long long bins,
                                                                          int nperm, const long long* __restrict__ blk,
                                                                          const long long* __restrict__ total,
                                                                          float* __restrict__ pool) {
    __shared__ long long sh[32];
    const long long first = (long long)blockIdx.x * NC_TILE + (long long)threadIdx.x * NC_ITEMS;
    long long unused;
    long long pos = blk[blockIdx.x] + block_exclusive_sum<long long>(nc_thread_count(q, bins, first), sh, &unused);
    const long long m = *total;
#pragma unroll
    for (int i = 0; i < NC_ITEMS; ++i) {
        const long long b = first + i;
        if (b < bins && (q == nullptr || q[b] == 0)) {
            for (int p = 0; p < nperm; ++p) pool[p * m + pos] = null_dist[p * bins + b];
            ++pos;
        }
    }
}

// ---------------------------------------------------------------- keyed subsampling
constexpr int FEISTEL_ROUNDS = 8;

// A pseudo-random permutation of [0, 2^(2h)): balanced Feistel network, round function = Philox4x32-10 keyed by the
// run seed with the trial in the counter.
__device__ __forceinline__ uint32_t feistel(uint32_t v, int h, uint64_t seed, uint32_t trial) {
    const uint32_t mask = (1u << h) - 1u;
    uint32_t L = v >> h, R = v & mask;
    Philox ph;
    ph.key0 = (uint32_t)seed;
    ph.key1 = (uint32_t)(seed >> 32);
#pragma unroll 1
    for (int r = 0; r < FEISTEL_ROUNDS; ++r) {
        ph.ctr[0] = R;
        ph.ctr[1] = (uint32_t)r;
        ph.ctr[2] = trial;
        ph.ctr[3] = 0x5EED5A3Du;
        ph.refill();
        const uint32_t F = ph.out[0] & mask;
        const uint32_t nl = R;
        R = L ^ F;
        L = nl;
    }
    return (L << h) | R;
}

__global__ void __launch_bounds__(256) null_subsample_kernel(const float* __restrict__ pool, long long n, int S,
                                                             int h, unsigned long long seed, int* __restrict__ idx_out,
                                                             float* __restrict__ samples) {
    const int t = blockIdx.y;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < S; i += (long long)gridDim.x * blockDim.x) {
        uint32_t v = (uint32_t)i;
        do {                                         // cycle walking: the orbit of i < n reaches [0, n) again
            v = feistel(v, h, seed, (uint32_t)t);
        } while ((long long)v >= n);
        if (idx_out != nullptr) idx_out[(long long)t * S + i] = (int)v;
        if (samples != nullptr) samples[(long long)t * S + i] = pool[v];
    }
}

// ---------------------------------------------------------------- generalized-normal MLE (scipy rv_continuous.fit)
constexpr int FIT_THREADS = 512;
constexpr double LOG_XMAX = 709.782712893384;      // numpy: log(finfo(float64).max), the _nnlf_and_penalty weight

struct FitShared {
    double sum[FIT_THREADS / 32];
    int bad[FIT_THREADS / 32];
    double result;
};

// Fixed-order block reduction of sum_i (a, b) over the CTA; every thread gets the totals.
__device__ __forceinline__ void block_sum2(double& a, int& b, FitShared& sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_down_sync(0xffffffffu, a, o);
        b += __shfl_down_sync(0xffffffffu, b, o);
    }
    if (lane == 0) {
        sh.sum[warp] = a;
        sh.bad[warp] = b;
    }
    __syncthreads();
    double s = 0.0;
    int nb = 0;
#pragma unroll
    for (int w = 0; w < FIT_THREADS / 32; ++w) {
        s += sh.sum[w];
        nb += sh.bad[w];
    }
    __syncthreads();
    a = s;
    b = nb;
}

// scipy's _penalized_nnlf for gennorm: -sum logpdf((x - loc) / scale, beta) + n log(scale), logpdf = log(beta / 2) -
// gammaln(1 / beta) - |z|^beta, with non-finite terms dropped and charged 100 log(XMAX) each.
__device__ double gennorm_nnlf(const float* __restrict__ x, int S, double beta, double loc, double scale, FitShared& sh) {
    if (!(beta > 0.0) || !(scale > 0.0)) return INFINITY;          // _argcheck / scale <= 0 (the same in every thread)
    const double ls = log2(scale);
    double acc = 0.0;
    int bad = 0;
    for (int i = threadIdx.x; i < S; i += FIT_THREADS) {
        const double t = fabs((double)__ldg(x + i) - loc);
        const double zb = t == 0.0 ? 0.0 : exp2(beta * (log2(t) - ls));    // |z|^beta
        if (zb < INFINITY) acc += zb;
        else ++bad;
    }
    block_sum2(acc, bad, sh);
    const double c = log(0.5 * beta) - lgamma(1.0 / beta);
    const double good = (double)(S - bad);
    double nll = -(good * c - acc);
    if (bad > 0) nll += (double)bad * LOG_XMAX * 100.0;
    return nll + (double)S * log(scale);
}

struct NelderMead {
    double sim[4][3];
    double fsim[4];
    int nfev;
    int iterations;
};

// numpy argsort of 4 values (insertion sort, i.e. stable) applied to the simplex
__device__ __forceinline__ void nm_sort(NelderMead& s) {
    for (int i = 1; i < 4; ++i)
        for (int j = i; j > 0 && s.fsim[j] < s.fsim[j - 1]; --j) {
            const double f = s.fsim[j];
            s.fsim[j] = s.fsim[j - 1];
            s.fsim[j - 1] = f;
            for (int k = 0; k < 3; ++k) {
                const double v = s.sim[j][k];
                s.sim[j][k] = s.sim[j - 1][k];
                s.sim[j - 1][k] = v;
            }
        }
}

// Point arithmetic without FMA contraction, as numpy evaluates it: a * u - b * w and a * u + b * w.
__device__ __forceinline__ void lincomb(double* out, double a, const double* u, double b, const double* w, bool minus) {
    for (int k = 0; k < 3; ++k) {
        const double p = __dmul_rn(a, u[k]), q = __dmul_rn(b, w[k]);
        out[k] = minus ? __dsub_rn(p, q) : __dadd_rn(p, q);
    }
}

__global__ void __launch_bounds__(FIT_THREADS) gennorm_fit_kernel(const float* __restrict__ samples, int S,
                                                                  double* __restrict__ params, int* __restrict__ status) {
    __shared__ FitShared sh;
    const float* x = samples + (long long)blockIdx.x * S;
    const int maxfun = 600, maxiter = 600;
    const double xatol = 1e-4, fatol = 1e-4;
    const double rho = 1.0, chi = 2.0, psi = 0.5, sigma = 0.5;

    // _fitstart: beta = 1 and the moment estimates fit_loc_scale gives for it (mean 0, variance 2 for beta = 1)
    double m = 0.0;
    int unused = 0;
    for (int i = threadIdx.x; i < S; i += FIT_THREADS) m += (double)x[i];
    block_sum2(m, unused, sh);
    const double mean = m / (double)S;
    double v = 0.0;
    for (int i = threadIdx.x; i < S; i += FIT_THREADS) {
        const double d = (double)x[i] - mean;
        v += d * d;
    }
    block_sum2(v, unused, sh);
    double shat = sqrt((v / (double)S) / 2.0);
    if (!(isfinite(shat) && shat > 0.0)) shat = 1.0;
    const double x0[3] = {1.0, isfinite(mean) ? mean : 0.0, shat};

    NelderMead s;
    for (int k = 0; k < 4; ++k) {
        for (int j = 0; j < 3; ++j) s.sim[k][j] = x0[j];
        s.fsim[k] = INFINITY;
    }
    for (int k = 0; k < 3; ++k) s.sim[k + 1][k] = x0[k] != 0.0 ? __dmul_rn(1.0 + 0.05, x0[k]) : 0.00025;
    s.nfev = 0;
    // the objective behind scipy's call counter: a call past maxfun raises instead of evaluating
    auto call = [&](const double* p, double& f) -> bool {
        if (s.nfev >= maxfun) return false;
        ++s.nfev;
        f = gennorm_nnlf(x, S, p[0], p[1], p[2], sh);
        return true;
    };
    for (int k = 0; k < 4; ++k)
        if (!call(s.sim[k], s.fsim[k])) break;
    nm_sort(s);
    s.iterations = 1;
    while (s.nfev < maxfun && s.iterations < maxiter) {
        bool done = true;                                        // max(...) <= tol, where a NaN fails the test
        for (int k = 1; k < 4; ++k) {
            for (int j = 0; j < 3; ++j) done = done && (fabs(s.sim[k][j] - s.sim[0][j]) <= xatol);
            done = done && (fabs(s.fsim[0] - s.fsim[k]) <= fatol);
        }
        if (done) break;
        double xbar[3];
        for (int j = 0; j < 3; ++j) xbar[j] = __ddiv_rn(__dadd_rn(__dadd_rn(s.sim[0][j], s.sim[1][j]), s.sim[2][j]), 3.0);
        bool aborted = false;
        double xr[3], fxr;
        lincomb(xr, 1.0 + rho, xbar, rho, s.sim[3], true);
        if (!call(xr, fxr)) {
            aborted = true;
        } else if (fxr < s.fsim[0]) {
            double xe[3], fxe;
            lincomb(xe, 1.0 + rho * chi, xbar, rho * chi, s.sim[3], true);
            if (!call(xe, fxe)) {
                aborted = true;
            } else if (fxe < fxr) {
                for (int j = 0; j < 3; ++j) s.sim[3][j] = xe[j];
                s.fsim[3] = fxe;
            } else {
                for (int j = 0; j < 3; ++j) s.sim[3][j] = xr[j];
                s.fsim[3] = fxr;
            }
        } else if (fxr < s.fsim[2]) {
            for (int j = 0; j < 3; ++j) s.sim[3][j] = xr[j];
            s.fsim[3] = fxr;
        } else {
            bool shrink = false;
            if (fxr < s.fsim[3]) {
                double xc[3], fxc;
                lincomb(xc, 1.0 + psi * rho, xbar, psi * rho, s.sim[3], true);
                if (!call(xc, fxc)) {
                    aborted = true;
                } else if (fxc <= fxr) {
                    for (int j = 0; j < 3; ++j) s.sim[3][j] = xc[j];
                    s.fsim[3] = fxc;
                } else {
                    shrink = true;
                }
            } else {
                double xcc[3], fxcc;
                lincomb(xcc, 1.0 - psi, xbar, psi, s.sim[3], false);
                if (!call(xcc, fxcc)) {
                    aborted = true;
                } else if (fxcc < s.fsim[3]) {
                    for (int j = 0; j < 3; ++j) s.sim[3][j] = xcc[j];
                    s.fsim[3] = fxcc;
                } else {
                    shrink = true;
                }
            }
            if (shrink)
                for (int k = 1; k < 4 && !aborted; ++k) {
                    for (int j = 0; j < 3; ++j)
                        s.sim[k][j] = __dadd_rn(s.sim[0][j], __dmul_rn(sigma, __dsub_rn(s.sim[k][j], s.sim[0][j])));
                    double f;
                    if (!call(s.sim[k], f)) aborted = true;      // the vertex has moved, its value has not
                    else s.fsim[k] = f;
                }
        }
        if (!aborted) ++s.iterations;
        nm_sort(s);
    }
    if (threadIdx.x == 0) {
        double fmin_ = s.fsim[0];
        for (int k = 1; k < 4; ++k) fmin_ = fmin(fmin_, s.fsim[k]);
        double* o = params + 4LL * blockIdx.x;
        o[0] = s.sim[0][0];
        o[1] = s.sim[0][1];
        o[2] = s.sim[0][2];
        o[3] = fmin_;
        status[2 * blockIdx.x] = s.iterations;
        status[2 * blockIdx.x + 1] = (s.nfev >= maxfun || s.iterations >= maxiter) ? 0 : 1;
    }
}

// ---------------------------------------------------------------- p-values
// Regularized upper incomplete gamma Q(a, z) for a in about [0.05, 20]: 1 - the power series of P for z < a + 1, the
// modified-Lentz continued fraction of Q otherwise; Q(a, 0) = 1 and Q(a, inf) = 0 exactly.
__device__ double gammaincc_dev(double a, double z) {
    if (z == 0.0) return 1.0;
    if (!(z < INFINITY)) return 0.0;
    const double lpre = a * log(z) - z - lgamma(a);
    const double eps = 1.1102230246251565e-16, tiny = 1e-300;
    if (z < a + 1.0) {
        double ap = a, del = 1.0 / a, sum = del;
        for (int n = 0; n < 1000; ++n) {
            ap += 1.0;
            del *= z / ap;
            sum += del;
            if (fabs(del) < fabs(sum) * eps) break;
        }
        const double q = 1.0 - sum * exp(lpre);
        return q < 0.0 ? 0.0 : q;
    }
    double b = z + 1.0 - a, c = 1.0 / tiny, d = 1.0 / b, h = d;
    for (int i = 1; i < 1000; ++i) {
        const double an = -i * (i - a);
        b += 2.0;
        d = an * d + b;
        if (fabs(d) < tiny) d = tiny;
        c = b + an / c;
        if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < eps) break;
    }
    const double q = exp(lpre) * h;
    return q > 1.0 ? 1.0 : q;
}

__global__ void __launch_bounds__(256) gennorm_pvalues_kernel(const float* __restrict__ x, long long n, double beta,
                                                              double loc, double scale, double* __restrict__ p) {
    const double a = 1.0 / beta;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double t = fabs((double)x[i] - loc) / scale;
        p[i] = gammaincc_dev(a, pow(t, beta));
    }
}

// ---------------------------------------------------------------- Benjamini-Hochberg
constexpr int RS_THREADS = 256, RS_ITEMS = 16, RS_TILE = RS_THREADS * RS_ITEMS, RS_WARPS = RS_THREADS / 32;

__global__ void __launch_bounds__(RS_THREADS) radix_hist_kernel(const unsigned long long* __restrict__ keys, long long n,
                                                                int shift, int nb, unsigned* __restrict__ hist) {
    __shared__ unsigned h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const long long base = (long long)blockIdx.x * RS_TILE;
#pragma unroll
    for (int i = 0; i < RS_ITEMS; ++i) {
        const long long e = base + i * RS_THREADS + threadIdx.x;
        if (e < n) atomicAdd(&h[(unsigned)(keys[e] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(long long)threadIdx.x * nb + blockIdx.x] = h[threadIdx.x];
}

// one block per digit: exclusive scan of that digit's per-tile counts, digit total out
__global__ void __launch_bounds__(1024) radix_scan_kernel(unsigned* __restrict__ hist, int nb,
                                                          unsigned* __restrict__ digit_total) {
    __shared__ unsigned sh[32];
    unsigned* row = hist + (long long)blockIdx.x * nb;
    const int per = (nb + blockDim.x - 1) / blockDim.x;
    const int lo = min(nb, per * (int)threadIdx.x), hi = min(nb, lo + per);
    unsigned s = 0;
    for (int i = lo; i < hi; ++i) s += row[i];
    unsigned all;
    unsigned run = block_exclusive_sum<unsigned>(s, sh, &all);
    for (int i = lo; i < hi; ++i) {
        const unsigned c = row[i];
        row[i] = run;
        run += c;
    }
    if (threadIdx.x == 0) digit_total[blockIdx.x] = all;
}

// Stable scatter of one tile: the elements of round i are base + i*256 + tid, ranked within their warp by match_any and
// across warps and rounds by per-digit counters, so equal digits keep their input order.
__global__ void __launch_bounds__(RS_THREADS) radix_scatter_kernel(const unsigned long long* __restrict__ keys_in,
                                                                   const int* __restrict__ idx_in, long long n, int shift,
                                                                   int nb, const unsigned* __restrict__ hist,
                                                                   const unsigned* __restrict__ digit_total,
                                                                   unsigned long long* __restrict__ keys_out,
                                                                   int* __restrict__ idx_out) {
    __shared__ unsigned base_of[256];
    __shared__ unsigned wcnt[RS_WARPS][256];
    __shared__ unsigned sh[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned all;
    const unsigned dbase = block_exclusive_sum<unsigned>(digit_total[tid], sh, &all);
    base_of[tid] = dbase + hist[(long long)tid * nb + blockIdx.x];
    for (int w = 0; w < RS_WARPS; ++w) wcnt[w][tid] = 0;
    __syncthreads();
    const long long base = (long long)blockIdx.x * RS_TILE;
    const unsigned lt = (1u << lane) - 1u;
    for (int i = 0; i < RS_ITEMS; ++i) {
        const long long e = base + i * RS_THREADS + tid;
        const bool valid = e < n;
        unsigned long long key = 0;
        int idx = 0;
        if (valid) {
            key = keys_in[e];
            idx = idx_in ? idx_in[e] : (int)e;
        }
        const unsigned d = valid ? (unsigned)(key >> shift) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const unsigned rank = __popc(peers & lt);
        if (valid && rank == 0) wcnt[warp][d] = __popc(peers);
        __syncthreads();
        if (valid) {
            unsigned pos = base_of[d] + rank;
            for (int w = 0; w < warp; ++w) pos += wcnt[w][d];
            keys_out[pos] = key;
            idx_out[pos] = idx;
        }
        __syncthreads();
        unsigned add = 0;
        for (int w = 0; w < RS_WARPS; ++w) {
            add += wcnt[w][tid];
            wcnt[w][tid] = 0;
        }
        base_of[tid] += add;
        __syncthreads();
    }
}

__device__ __forceinline__ double bh_raw(const unsigned long long* keys, long long i, long long n) {
    return __ddiv_rn(__longlong_as_double((long long)keys[i]), __ddiv_rn((double)(i + 1), (double)n));
}

__global__ void __launch_bounds__(RS_THREADS) bh_block_min_kernel(const unsigned long long* __restrict__ keys, long long n,
                                                                  double* __restrict__ bmin) {
    __shared__ double sh[32];
    const long long first = (long long)blockIdx.x * RS_TILE + (long long)threadIdx.x * RS_ITEMS;
    double m = INFINITY;
    for (int i = 0; i < RS_ITEMS; ++i)
        if (first + i < n) m = fmin(m, bh_raw(keys, first + i, n));
    const double after = block_exclusive_suffix_min(m, sh);
    if (threadIdx.x == 0) bmin[blockIdx.x] = fmin(m, after);
}

// one block: bmin[b] <- minimum over the tiles after b
__global__ void __launch_bounds__(1024) bh_carry_kernel(double* __restrict__ bmin, int nb) {
    __shared__ double sh[32];
    const int per = (nb + blockDim.x - 1) / blockDim.x;
    const int lo = min(nb, per * (int)threadIdx.x), hi = min(nb, lo + per);
    double m = INFINITY;
    for (int i = lo; i < hi; ++i) m = fmin(m, bmin[i]);
    double run = block_exclusive_suffix_min(m, sh);
    for (int i = hi - 1; i >= lo; --i) {
        const double c = bmin[i];
        bmin[i] = run;
        run = fmin(run, c);
    }
}

__global__ void __launch_bounds__(RS_THREADS) bh_apply_kernel(const unsigned long long* __restrict__ keys,
                                                              const int* __restrict__ idx, long long n,
                                                              const double* __restrict__ carry, double* __restrict__ q) {
    __shared__ double sh[32];
    const long long first = (long long)blockIdx.x * RS_TILE + (long long)threadIdx.x * RS_ITEMS;
    double m = INFINITY;
    for (int i = 0; i < RS_ITEMS; ++i)
        if (first + i < n) m = fmin(m, bh_raw(keys, first + i, n));
    double run = fmin(block_exclusive_suffix_min(m, sh), carry[blockIdx.x]);
    for (int i = RS_ITEMS - 1; i >= 0; --i) {
        const long long e = first + i;
        if (e >= n) continue;
        run = fmin(run, bh_raw(keys, e, n));
        q[idx[e]] = run > 1.0 ? 1.0 : run;
    }
}

struct BhLayout {
    size_t keys_a, keys_b, idx_a, idx_b, hist, totals, bmin, bytes;
    int nb;
};

static BhLayout bh_layout(int64_t n) {
    BhLayout L;
    L.nb = (int)((n + RS_TILE - 1) / RS_TILE);
    size_t off = 0;
    auto take = [&](size_t b) {
        const size_t o = off;
        off += align256(b);
        return o;
    };
    L.keys_a = take((size_t)n * 8);
    L.keys_b = take((size_t)n * 8);
    L.idx_a = take((size_t)n * 4);
    L.idx_b = take((size_t)n * 4);
    L.hist = take((size_t)256 * L.nb * 4);
    L.totals = take(256 * 4);
    L.bmin = take((size_t)L.nb * 8);
    L.bytes = off;
    return L;
}

}  // namespace epi

using namespace epi;

extern "C" int epi_null_compact_workspace_size(int64_t bins, int64_t* bytes_out) {
    EPI_REQUIRE(bins >= 0 && bytes_out != nullptr, "bad argument");
    *bytes_out = (int64_t)align256(((size_t)(bins + NC_TILE - 1) / NC_TILE + 1) * sizeof(long long));
    return 0;
}

extern "C" int epi_null_compact(const float* null_dev, const uint8_t* quiescent_dev, int64_t bins, int32_t nperm,
                                float* pool_out, int64_t* count_out_dev, void* workspace, int64_t workspace_bytes,
                                void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && nperm >= 1, "bad null shape");
    EPI_REQUIRE(count_out_dev != nullptr, "null pointer argument");
    if (bins == 0) {
        EPI_CUDA(cudaMemsetAsync(count_out_dev, 0, sizeof(int64_t), st));
        return 0;
    }
    int64_t need = 0;
    epi_null_compact_workspace_size(bins, &need);
    EPI_REQUIRE(null_dev && pool_out && workspace, "null pointer argument");
    EPI_REQUIRE(workspace_bytes >= need, "workspace of %lld bytes, need %lld", (long long)workspace_bytes, (long long)need);
    const long long nblk = (bins + NC_TILE - 1) / NC_TILE;
    EPI_REQUIRE(nblk < (1LL << 31), "too many bins");
    long long* blk = static_cast<long long*>(workspace);
    long long* total = reinterpret_cast<long long*>(count_out_dev);
    null_compact_count_kernel<<<(unsigned)nblk, NC_THREADS, 0, st>>>(quiescent_dev, bins, blk);
    exclusive_scan_ll_kernel<<<1, 1024, 0, st>>>(blk, nblk, total);
    null_compact_scatter_kernel<<<(unsigned)nblk, NC_THREADS, 0, st>>>(null_dev, quiescent_dev, bins, nperm, blk, total,
                                                                       pool_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_null_subsample(const float* pool_dev, int64_t n, int32_t trials, int32_t size, uint64_t seed,
                                  int32_t* idx_out, float* samples_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(n >= 1 && n < (1LL << 31), "pool size %lld out of range [1, 2^31)", (long long)n);
    EPI_REQUIRE(trials >= 1 && trials <= 65535 && size >= 1 && size <= n,
                "need 1 <= trials <= 65535 and 1 <= size <= pool size (%d, %d, %lld)", trials, size, (long long)n);
    EPI_REQUIRE(idx_out || samples_out, "no output requested");
    EPI_REQUIRE(samples_out == nullptr || pool_dev != nullptr, "null pointer argument");
    int bits = 1;
    while ((1LL << bits) < n) ++bits;
    const int h = (bits + 1) / 2;                         // 2^(2h) < 4n: under four Feistel walks per index on average
    dim3 grid((unsigned)std::min<long long>((size + 255) / 256, 4096), (unsigned)trials);
    null_subsample_kernel<<<grid, 256, 0, st>>>(pool_dev, n, size, h, (unsigned long long)seed, idx_out, samples_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_gennorm_fit(const float* samples_dev, int32_t trials, int32_t size, double* params_out,
                               int32_t* status_out, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(trials >= 1 && size >= 1, "bad fit shape (%d trials of %d points)", trials, size);
    EPI_REQUIRE(samples_dev && params_out && status_out, "null pointer argument");
    gennorm_fit_kernel<<<(unsigned)trials, FIT_THREADS, 0, st>>>(samples_dev, size, params_out, status_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_gennorm_pvalues(const float* x_dev, int64_t n, double beta, double loc, double scale, double* p_out,
                                   void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(n >= 0, "bad shape");
    EPI_REQUIRE(beta > 0.0 && scale > 0.0 && isfinite(beta) && isfinite(scale) && isfinite(loc),
                "gennorm parameters out of range (beta=%g loc=%g scale=%g)", beta, loc, scale);
    if (n == 0) return 0;
    EPI_REQUIRE(x_dev && p_out, "null pointer argument");
    gennorm_pvalues_kernel<<<grid_for_n(n, 256, 16), 256, 0, st>>>(x_dev, n, beta, loc, scale, p_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_bh_workspace_size(int64_t n, int64_t* bytes_out) {
    EPI_REQUIRE(n >= 0 && n < (1LL << 31) && bytes_out != nullptr, "bad argument");
    *bytes_out = (int64_t)bh_layout(n).bytes;
    return 0;
}

extern "C" int epi_bh_adjust(const double* p_dev, int64_t n, double* q_out, void* workspace, int64_t workspace_bytes,
                             void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(n >= 0 && n < (1LL << 31), "%lld p-values: the index payload is 32-bit", (long long)n);
    if (n == 0) return 0;
    const BhLayout L = bh_layout(n);
    EPI_REQUIRE(p_dev && q_out && workspace, "null pointer argument");
    EPI_REQUIRE(workspace_bytes >= (int64_t)L.bytes, "workspace of %lld bytes, need %lld", (long long)workspace_bytes,
                (long long)L.bytes);
    char* ws = static_cast<char*>(workspace);
    unsigned long long* kbuf[2] = {reinterpret_cast<unsigned long long*>(ws + L.keys_a),
                                   reinterpret_cast<unsigned long long*>(ws + L.keys_b)};
    int* ibuf[2] = {reinterpret_cast<int*>(ws + L.idx_a), reinterpret_cast<int*>(ws + L.idx_b)};
    unsigned* hist = reinterpret_cast<unsigned*>(ws + L.hist);
    unsigned* totals = reinterpret_cast<unsigned*>(ws + L.totals);
    double* bmin = reinterpret_cast<double*>(ws + L.bmin);
    // p >= 0, so the IEEE bit patterns sort like the values
    const unsigned long long* kin = reinterpret_cast<const unsigned long long*>(p_dev);
    const int* iin = nullptr;                              // first pass: the payload is the element index
    int cur = 0;
    for (int shift = 0; shift < 64; shift += 8) {
        radix_hist_kernel<<<L.nb, RS_THREADS, 0, st>>>(kin, n, shift, L.nb, hist);
        radix_scan_kernel<<<256, 1024, 0, st>>>(hist, L.nb, totals);
        radix_scatter_kernel<<<L.nb, RS_THREADS, 0, st>>>(kin, iin, n, shift, L.nb, hist, totals, kbuf[cur], ibuf[cur]);
        kin = kbuf[cur];
        iin = ibuf[cur];
        cur ^= 1;
    }
    bh_block_min_kernel<<<L.nb, RS_THREADS, 0, st>>>(kin, n, bmin);
    bh_carry_kernel<<<1, 1024, 0, st>>>(bmin, L.nb);
    bh_apply_kernel<<<L.nb, RS_THREADS, 0, st>>>(kin, iin, n, bmin, q_out);
    EPI_CUDA(cudaGetLastError());
    return 0;
}
