// K6 -- S3 scores.
//
// Reference (scores.py:455-506, s3Score): scoreArrOnes = klScoreND(ones/(C(C-1)), E3) is a [C][C][K][K] table of
// pair terms T[i][j][a][c] = q log2(q / E3[i][j][a][c]), q = 1/(C(C-1)) (0 where E3 == 0), and per bin
//      score[b][s] = sum over ordered pairs i != j with x[b][j] == s of T[i][j][x[b][i]][x[b][j]]
// (np.add.at buckets by the state of the SECOND biosample of the pair).  The reference evaluates the table and
// the 693 k-term sums in float32; this kernel evaluates both in float64 -- it is held to the float64
// restatement (oracle s3_scores_f64) at 1e-9 and agrees with the reference's float32 result to the
// reference's own accumulation noise (SURVEY.md section 8c).
//
// The work is C(C-1) table look-ups per bin (8.7e11 for chr1 at 833 biosamples) into a 1.8 GB table: neither
// HBM- nor tensor-shaped.  Blocking (version 2; version 1 gathered through L1 at 1.8e11 look-ups/s):
//   * a CTA owns BC = 256*BPT consecutive bins (BPT per thread) and walks j in blocks of JC biosamples; for a
//     j-block it keeps JC*BPT float64 accumulators per thread in registers and runs over all i;
//   * for every (i, j-block) the JC consecutive K*K term blocks T[i][j0..j0+JC) are ONE contiguous slab, streamed
//     into a two-stage shared-memory ring by a producer warp with 1D bulk copies (cp.async.bulk + mbarrier), so the
//     look-ups are LDS.64 (identical (a,c) pairs across lanes -- the common case in real data -- broadcast);
//   * labels come from a transposed copy xT[C][bins] so a thread's BPT labels of biosample i are one coalesced load;
//   * per-bin score rows live in shared memory and are written once: no atomics, deterministic summation order.
// T is streamed once per CTA: L2->SM traffic = (bins / BC) * 1.8 GB.
//
// Symmetry (version 3): the expected table of s3Calc is symmetric, E3[i][j][a][c] == E3[j][i][c][a], hence so are the
// terms, and the ordered pairs (i,j) and (j,i) of a bin contribute the SAME value -- once to the bucket of x_j, once to
// the bucket of x_i.  The SYM kernel walks only i < j: one look-up per UNORDERED pair, added to the j accumulator in
// registers and, summed over the j-block, to the score row of x_i in shared memory: half the look-ups (the limiter) and
// half the slab traffic.  s3_symmetry_kernel verifies the property on the device for every table it is given (a foreign
// exp_freq file need not have it); both kernels are queued and the one that does not apply exits at once.
#include "common.cuh"

namespace epi {

constexpr int S3S_THREADS = 256;          // consumer threads (+ 32 producer threads)
constexpr int S3S_JC = 8;                 // biosamples per j-block

__host__ __device__ inline long long s3_block_stride(int K) { return ((long long)K * K + 1) & ~1ll; }   // 16-byte blocks

// terms in padded block layout: block (i*C + j) holds K*K doubles [a][c] (+ pad), S3S_JC zero blocks at the end
// (the last slab of a row starts at most S3S_JC - 1 blocks before the end of the row)
__global__ void __launch_bounds__(256) s3_terms_kernel(const float* __restrict__ e3, int cols, int K, double q,
                                                       double* __restrict__ terms, long long nblocks_total) {
    const long long blk = s3_block_stride(K);
    const long long kk = (long long)K * K;
    const long long n = nblocks_total * blk;
    const long long nreal = (long long)cols * cols;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / blk, r = idx - b * blk;
        double v = 0.0;
        if (b < nreal && r < kk) {
            const double e = (double)e3[b * kk + r];
            v = (e == 0.0) ? 0.0 : q * log2(q / e);          // klScoreND masks (scores.py:550); q > 0 always
        }
        terms[idx] = v;
    }
}

// x[bins][pitch] -> xT[cols][bp] (bins >= `bins` filled with label 0)
__global__ void __launch_bounds__(256) s3_transpose_kernel(const int8_t* __restrict__ x, long long bins, int cols,
                                                           long long pitch, uint8_t* __restrict__ xt, long long bp) {
    __shared__ uint8_t tile[64][65];
    const long long b0 = (long long)blockIdx.x * 64;
    const int j0 = blockIdx.y * 64;
    for (int i = threadIdx.x; i < 64 * 64; i += 256) {
        const int r = i >> 6, c = i & 63;                   // r: bin, c: column (coalesced along columns)
        uint8_t v = 0;
        if (b0 + r < bins && j0 + c < cols) v = (uint8_t)x[(b0 + r) * pitch + j0 + c];
        tile[r][c] = v;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 64 * 64; i += 256) {
        const int c = i >> 6, r = i & 63;                   // coalesced along bins
        if (j0 + c < cols && b0 + r < bp) xt[(long long)(j0 + c) * bp + b0 + r] = tile[r][c];
    }
}

// *flag = 0 if some T[i][j][a][c] != T[j][i][c][a] (bit pattern compare; the flag is preset to non-zero by the caller)
__global__ void __launch_bounds__(256) s3_symmetry_kernel(const double* __restrict__ terms, int cols, int K,
                                                          int* __restrict__ flag) {
    const long long blk = s3_block_stride(K);
    const long long kk = (long long)K * K;
    const long long n = (long long)cols * cols * kk;
    bool bad = false;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long pair = idx / kk;
        const int r = (int)(idx - pair * kk);
        const int i = (int)(pair / cols), j = (int)(pair - (long long)i * cols);
        if (i < j) {
            const int a = r / K, c = r - a * K;
            const long long v = __double_as_longlong(terms[pair * blk + r]);
            const long long w = __double_as_longlong(terms[((long long)j * cols + i) * blk + (long long)c * K + a]);
            bad |= v != w;
        }
    }
    if (bad) *flag = 0;
}

// SYM: 0 = all ordered pairs (any table), 1 = unordered pairs of a symmetric table.  *gate != 0 means symmetric: only the
// kernel that applies does the work, the other one exits at once.
template <int BPT, int JC, int SYM>
__global__ void __launch_bounds__(S3S_THREADS + 32, 1)
s3_score_kernel(const uint8_t* __restrict__ xt, long long bp, long long bins, int cols, int K,
                const double* __restrict__ terms, const int* __restrict__ gate, int nslab, float* __restrict__ out32,
                double* __restrict__ out64) {
    if ((*gate != 0) != (SYM != 0)) return;
    constexpr int BC = S3S_THREADS * BPT;
    extern __shared__ __align__(128) uint8_t smem[];
    const int blk = (int)s3_block_stride(K);
    const int slab_bytes = JC * blk * 8;
    // score rows: sc[(u * 256 + tid) * KP + state], KP odd, so that the lanes of a warp hit different banks when they
    // update the same state (the SYM kernel read-modify-writes one row entry per bin and slab)
    const int KP = K | 1;
    double* sc = reinterpret_cast<double*>(smem);                                   // [BPT][256][KP]
    uint8_t* slabs = smem + (((size_t)BC * KP * 8 + 127) & ~(size_t)127);          // nslab slabs
    uint64_t* full = reinterpret_cast<uint64_t*>(slabs + (size_t)nslab * slab_bytes);
    uint64_t* empty = full + nslab;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < nslab; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], S3S_THREADS / 32);
        }
        mbar_fence_init();
    }
    for (int i = tid; i < BC * KP; i += blockDim.x) sc[i] = 0.0;
    __syncthreads();

    const int njb = (cols + JC - 1) / JC;
    if (warp == S3S_THREADS / 32) {
        // ---------------- producer: stream the term slabs (i, j-block) ----------------
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int jb = 0; jb < njb; ++jb) {
                const int iend = SYM ? ((jb + 1) * JC < cols ? (jb + 1) * JC : cols) : cols;
                for (int i = 0; i < iend; ++i) {
                    mbar_wait(&empty[s], ph ^ 1);
                    mbar_expect_tx(&full[s], slab_bytes);
                    bulk_load_1d(slabs + (size_t)s * slab_bytes, terms + ((long long)i * cols + jb * JC) * blk,
                                 slab_bytes, &full[s]);
                    if (++s == nslab) {
                        s = 0;
                        ph ^= 1;
                    }
                }
            }
        }
        return;
    }

    // ---------------- consumers: BPT bins per thread ----------------
    const long long bin0 = (long long)blockIdx.x * BC + (long long)tid * BPT;
    const uint8_t* col = xt + bin0;                          // + i * bp
    double* my_sc = sc + (size_t)tid * KP;                  // + u * 256 * KP
    const uint32_t slab0 = smem_u32(slabs);
    int s = 0;
    uint32_t ph = 0;

    auto load_labels = [&](int i, uint32_t (&lab)[BPT]) {
        if constexpr (BPT == 4) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(col + (long long)i * bp);
            lab[0] = w & 0xff; lab[1] = (w >> 8) & 0xff; lab[2] = (w >> 16) & 0xff; lab[3] = w >> 24;
        } else if constexpr (BPT == 2) {
            const uint32_t w = *reinterpret_cast<const uint16_t*>(col + (long long)i * bp);
            lab[0] = w & 0xff; lab[1] = w >> 8;
        } else {
#pragma unroll
            for (int u = 0; u < BPT; ++u) lab[u] = col[(long long)i * bp + u];
        }
    };

    for (int jb = 0; jb < njb; ++jb) {
        const int j0 = jb * JC;
        uint32_t off[BPT][JC];       // byte offset of (jj, c) inside a slab
        uint32_t cst[BPT][JC];       // state of biosample j0+jj in bin u
        double acc[BPT][JC];
#pragma unroll
        for (int jj = 0; jj < JC; ++jj) {
            uint32_t lab[BPT];
            load_labels(j0 + jj < cols ? j0 + jj : cols - 1, lab);
#pragma unroll
            for (int u = 0; u < BPT; ++u) {
                cst[u][jj] = lab[u];
                off[u][jj] = (uint32_t)(jj * blk + (int)lab[u]) * 8u;
                acc[u][jj] = 0.0;
            }
        }
        uint32_t nxt[BPT];
        load_labels(0, nxt);
        const int iend = SYM ? (j0 + JC < cols ? j0 + JC : cols) : cols;
        const int njv = cols - j0 < JC ? cols - j0 : JC;          // biosamples of this j-block that exist
        for (int i = 0; i < iend; ++i) {
            uint32_t a[BPT], ai[BPT];
#pragma unroll
            for (int u = 0; u < BPT; ++u) {
                ai[u] = nxt[u];
                a[u] = nxt[u] * (uint32_t)(K * 8);
            }
            if (i + 1 < iend) load_labels(i + 1, nxt);          // prefetch the next biosample's labels
            mbar_wait(&full[s], ph);
            const uint32_t base = slab0 + (uint32_t)s * (uint32_t)slab_bytes;
            const bool diag = (i >= j0) && (i < j0 + JC);
            double dep = 0.0;                                    // the last value read from the slab (see mbar_arrive_after)
            if (SYM) {
                // unordered pairs i < j: the term goes to the bucket of x_j (registers) and to the bucket of x_i (score row)
#pragma unroll
                for (int u = 0; u < BPT; ++u) {
                    double si = 0.0;
#pragma unroll
                    for (int jj = 0; jj < JC; ++jj) {
                        if (jj < njv && (!diag || j0 + jj > i)) {      // real biosample, and j > i inside the diagonal block
                            double t;
                            asm volatile("ld.shared.f64 %0, [%1];" : "=d"(t) : "r"(base + a[u] + off[u][jj]));
                            acc[u][jj] += t;
                            si += t;
                            dep = t;
                        }
                    }
                    my_sc[(size_t)u * S3S_THREADS * KP + ai[u]] += si;
                }
            } else if (!diag) {
#pragma unroll
                for (int u = 0; u < BPT; ++u) {
#pragma unroll
                    for (int jj = 0; jj < JC; ++jj) {
                        double t;
                        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(t) : "r"(base + a[u] + off[u][jj]));
                        acc[u][jj] += t;
                        dep = t;
                    }
                }
            } else {
#pragma unroll
                for (int u = 0; u < BPT; ++u) {
#pragma unroll
                    for (int jj = 0; jj < JC; ++jj) {
                        if (i != j0 + jj) {                      // the pair (i, i) does not exist
                            double t;
                            asm volatile("ld.shared.f64 %0, [%1];" : "=d"(t) : "r"(base + a[u] + off[u][jj]));
                            acc[u][jj] += t;
                            dep = t;
                        }
                    }
                }
            }
            __syncwarp();
            // The slab goes back to the producer only after its look-ups have returned.  SYM: the read-modify-write of the
            // score row above depends on every loaded term and precedes the arrive in program order.  Ordered-pair kernel:
            // the arrive takes the last loaded value as an operand (mbar_arrive_after, common.cuh).
            if (lane == 0) mbar_arrive_after(&empty[s], dep);
            if (++s == nslab) {
                s = 0;
                ph ^= 1;
            }
        }
        // bucket by the state of the second biosample (np.add.at index dataArr[row, J], scores.py:496)
#pragma unroll
        for (int jj = 0; jj < JC; ++jj) {
            if (j0 + jj < cols) {
#pragma unroll
                for (int u = 0; u < BPT; ++u) my_sc[(size_t)u * S3S_THREADS * KP + cst[u][jj]] += acc[u][jj];
            }
        }
    }
    // ---------------- write the CTA's score rows ----------------
    asm volatile("bar.sync 1, %0;" ::"r"(S3S_THREADS) : "memory");      // consumers only (the producer warp has left)
    const long long cta_bin0 = (long long)blockIdx.x * BC;
    const long long nvalid = (bins - cta_bin0) < BC ? (bins - cta_bin0) : BC;
    for (long long i = tid; i < nvalid * K; i += S3S_THREADS) {
        const int lb = (int)(i / K), st = (int)(i - (long long)lb * K);         // local bin = owner thread * BPT + u
        const double v = sc[((size_t)(lb % BPT) * S3S_THREADS + lb / BPT) * KP + st];
        if (out32 != nullptr) out32[cta_bin0 * K + i] = (float)v;
        if (out64 != nullptr) out64[cta_bin0 * K + i] = v;
    }
}

template <int BPT, int JC>
static int launch_s3_score(const uint8_t* xt, int64_t bp, int64_t bins, int cols, int K, const double* terms,
                           const int* gate, float* o32, double* o64, cudaStream_t st) {
    constexpr int BC = S3S_THREADS * BPT;
    const size_t slab = (size_t)JC * s3_block_stride(K) * 8;
    const size_t rows = (((size_t)BC * (K | 1) * 8 + 127) & ~(size_t)127);
    const int nslab = rows + 4 * slab + 128 <= 224 * 1024 ? 4 : (rows + 3 * slab + 128 <= 224 * 1024 ? 3 : 2);
    const size_t smem = rows + (size_t)nslab * slab + 128;
    auto sym = s3_score_kernel<BPT, JC, 1>;
    auto full = s3_score_kernel<BPT, JC, 0>;
    EPI_CUDA(cudaFuncSetAttribute(sym, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    EPI_CUDA(cudaFuncSetAttribute(full, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)((bins + BC - 1) / BC);
    sym<<<grid, S3S_THREADS + 32, smem, st>>>(xt, bp, bins, cols, K, terms, gate, nslab, o32, o64);
    full<<<grid, S3S_THREADS + 32, smem, st>>>(xt, bp, bins, cols, K, terms, gate, nslab, o32, o64);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace epi

using namespace epi;

extern "C" int epi_s3_terms_size(int32_t cols, int32_t K, int64_t* doubles_out) {
    EPI_REQUIRE(cols >= 2 && K >= 1 && K <= EPI_MAX_STATES && doubles_out != nullptr, "bad S3 shape");
    *doubles_out = ((int64_t)cols * cols + S3S_JC) * s3_block_stride(K);
    return 0;
}

extern "C" int epi_s3_terms(const float* exp3_dev, int32_t cols, int32_t K, double* terms_dev, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(cols >= 2 && K >= 1 && K <= EPI_MAX_STATES, "bad S3 shape (needs at least 2 biosamples)");
    EPI_REQUIRE(exp3_dev != nullptr && terms_dev != nullptr, "null pointer argument");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(terms_dev) & 15) == 0, "terms_dev must be 16-byte aligned");
    const long long nblocks = (long long)cols * cols + S3S_JC;
    const long long n = nblocks * s3_block_stride(K);
    const double q = 1.0 / ((double)cols * (double)(cols - 1));
    long long blocks = (n + 255) / 256;
    const long long cap = (long long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    s3_terms_kernel<<<(unsigned)blocks, 256, 0, st>>>(exp3_dev, cols, K, q, terms_dev, nblocks);
    EPI_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int epi_scores_s3(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t K,
                             const double* terms_dev, float* out32_dev, double* out64_dev, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 0 && cols >= 2 && pitch >= cols && K >= 1 && K <= EPI_MAX_STATES, "bad S3 shape");
    if (bins == 0 || (out32_dev == nullptr && out64_dev == nullptr)) return 0;
    EPI_REQUIRE(x_dev != nullptr && terms_dev != nullptr, "null pointer argument");
    EPI_REQUIRE((reinterpret_cast<uintptr_t>(terms_dev) & 15) == 0, "terms_dev must be 16-byte aligned");
    // choose the bins per thread so that score rows BC*K*8 + two slabs JC*blk*8 fit 220 KB of shared memory.  JC = 8 fits
    // at BPT = 1 for every K <= 32 (66 KB of rows + 128 KB of slabs at K = 32); the check guards a larger EPI_MAX_STATES.
    const size_t blk8 = (size_t)s3_block_stride(K) * 8;
    int bpt = 4;
    auto fits = [&](int b) { return (size_t)S3S_THREADS * b * (K | 1) * 8 + 2 * (size_t)S3S_JC * blk8 + 256 <= 220 * 1024; };
    if (bins <= S3S_THREADS * 2) bpt = bins <= S3S_THREADS ? 1 : 2;              // small inputs: more CTAs
    while (!fits(bpt) && bpt > 1) bpt >>= 1;
    EPI_REQUIRE(fits(bpt), "S3 score blocking does not fit shared memory for K=%d", K);
    DeviceWorkspace* ws = device_workspace();
    EPI_REQUIRE(ws != nullptr, "could not allocate the per-device workspace");
    const int64_t bc = (int64_t)S3S_THREADS * bpt;
    const int64_t bp = ((bins + bc - 1) / bc) * bc;
    uint8_t* xt = nullptr;
    EPI_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&xt), (size_t)(bp * cols), st));
    dim3 tg((unsigned)((bp + 63) / 64), (unsigned)((cols + 63) / 64));
    s3_transpose_kernel<<<tg, 256, 0, st>>>(x_dev, bins, cols, pitch, xt, bp);
    // is the table symmetric (it is whenever it comes from s3Calc)?  decided on the device, no host round trip
    int* gate = &ws->s3_symmetric;
    EPI_CUDA(cudaMemsetAsync(gate, 1, 4, st));
    s3_symmetry_kernel<<<sm_count() * 8, 256, 0, st>>>(terms_dev, cols, K, gate);
    int rc = 0;
#define EPI_S3S_CASE(B) if (bpt == B) rc = launch_s3_score<B, S3S_JC>(xt, bp, bins, cols, K, terms_dev, gate, out32_dev, out64_dev, st); else
    EPI_S3S_CASE(4) EPI_S3S_CASE(2) EPI_S3S_CASE(1) { set_error("no S3 score kernel for %d bins per thread", bpt); rc = 2; }
#undef EPI_S3S_CASE
    cudaFreeAsync(xt, st);
    return rc;
}
