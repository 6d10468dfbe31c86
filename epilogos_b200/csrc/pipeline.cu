// epi_single_host: the whole S1/S2 path for one in-memory matrix held in HOST memory -- what
// expected.main -> expectedCombination.main -> scores.main compute (run.py:196, 231, 246), without the
// TSV / gzip I/O.  H2D copies of the matrix are chunked on a copy stream and overlapped with the count
// kernel; the score kernel runs chunk by chunk so its D2H copies overlap as well.
#include <mutex>

#include "common.cuh"

namespace epi {

struct HostPipe {
    cudaStream_t copy = nullptr, compute = nullptr, d2h = nullptr;     // H2D, kernels, D2H: one stream each
    cudaEvent_t copied[2] = {nullptr, nullptr}, counted[2] = {nullptr, nullptr}, scored[2] = {nullptr, nullptr},
                d2h_done[2] = {nullptr, nullptr};
    int8_t* xbuf[2] = {nullptr, nullptr};
    size_t xbuf_bytes = 0;
    uint8_t* pbuf[2] = {nullptr, nullptr};     // packed chunks (bit-packed transport layout)
    size_t pbuf_bytes = 0;
    uint16_t* cnt = nullptr;
    size_t cnt_bytes = 0;
    float* scores[2] = {nullptr, nullptr};
    size_t score_bytes = 0;
    int64_t* tables = nullptr;     // n (int64 K*K) followed by exp (float K*K)
    int device = -1;
};

static HostPipe g_pipe;
static std::mutex g_pipe_mutex;

static int ensure(void** p, size_t* have, size_t want) {
    if (*have >= want) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *have = 0;
    EPI_CUDA(cudaMalloc(p, want));
    *have = want;
    return 0;
}

static int pipe_init(HostPipe& hp) {
    int dev = 0;
    EPI_CUDA(cudaGetDevice(&dev));
    if (hp.device == dev) return 0;
    EPI_REQUIRE(hp.device == -1, "epi_single_host was first used on device %d; it keeps one workspace per process",
                hp.device);
    EPI_CUDA(cudaStreamCreateWithFlags(&hp.copy, cudaStreamNonBlocking));
    EPI_CUDA(cudaStreamCreateWithFlags(&hp.compute, cudaStreamNonBlocking));
    EPI_CUDA(cudaStreamCreateWithFlags(&hp.d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        EPI_CUDA(cudaEventCreateWithFlags(&hp.d2h_done[i], cudaEventDisableTiming));
        EPI_CUDA(cudaEventCreateWithFlags(&hp.copied[i], cudaEventDisableTiming));
        EPI_CUDA(cudaEventCreateWithFlags(&hp.counted[i], cudaEventDisableTiming));
        EPI_CUDA(cudaEventCreateWithFlags(&hp.scored[i], cudaEventDisableTiming));
    }
    EPI_CUDA(cudaMalloc(reinterpret_cast<void**>(&hp.tables),
                        (size_t)EPI_MAX_STATES * EPI_MAX_STATES * (sizeof(int64_t) + sizeof(float))));
    hp.device = dev;
    return 0;
}

}  // namespace epi

using namespace epi;

// bits == 0: x_host is the int8 matrix (row pitch `pitch`); bits == 4 / 5: x_host is the bit-packed transport layout
// (csrc/packbits.cu, row pitch `pitch`), expanded on the device chunk by chunk right before the count kernel.
static int single_host_impl(const uint8_t* x_host, int64_t bins, int32_t cols, int64_t pitch, int32_t bits, int32_t K,
                            int32_t saliency, int64_t* counts_host, float* exp_host, float* scores_host) {
    if (check_device()) return 3;
    EPI_REQUIRE(saliency == 1 || saliency == 2, "epi_single_host handles saliency 1 and 2 (got %d)", saliency);
    EPI_REQUIRE(bins >= 1 && bins < (1ll << 31), "bins=%lld out of range", (long long)bins);
    EPI_REQUIRE(cols >= (saliency == 2 ? 2 : 1) && cols <= 65535, "cols=%d out of range", cols);
    EPI_REQUIRE(bits == 0 || bits == 4 || bits == 5, "bits=%d: int8 (0) or 4 / 5 bits per label", bits);
    if (bits == 0) EPI_REQUIRE(pitch >= cols, "pitch=%lld smaller than cols=%d", (long long)pitch, cols);
    else EPI_REQUIRE(pitch >= (int64_t)((cols + 7) / 8) * bits && (pitch & 15) == 0, "packed pitch %lld must be a multiple of "
                     "16 and hold %d labels of %d bits (epi_packed_pitch)", (long long)pitch, cols, bits);
    EPI_REQUIRE(K >= 1 && K <= EPI_MAX_STATES, "num_states=%d out of range [1, %d]", K, EPI_MAX_STATES);
    EPI_REQUIRE(bits == 0 || K <= (1 << bits), "%d states do not fit %d bits per label", K, bits);
    EPI_REQUIRE(x_host != nullptr, "null matrix pointer");

    std::lock_guard<std::mutex> lock(g_pipe_mutex);
    HostPipe& hp = g_pipe;
    if (int rc = pipe_init(hp)) return rc;

    const int64_t dpitch = ((int64_t)cols + 15) & ~15ll;
    int64_t chunk = (int64_t)(192ll << 20) / dpitch;           // ~192 MB of matrix per chunk
    chunk = (chunk / 4096) * 4096;
    if (chunk < 4096) chunk = 4096;
    if (chunk > bins) chunk = bins;
    const int64_t nchunks = (bins + chunk - 1) / chunk;
    const int ntab = saliency == 1 ? K : K * K;

    size_t xb = hp.xbuf_bytes;
    if (int rc = ensure(reinterpret_cast<void**>(&hp.xbuf[0]), &xb, (size_t)(chunk * dpitch))) return rc;
    if (int rc = ensure(reinterpret_cast<void**>(&hp.xbuf[1]), &hp.xbuf_bytes, (size_t)(chunk * dpitch))) return rc;
    if (int rc = ensure(reinterpret_cast<void**>(&hp.cnt), &hp.cnt_bytes, (size_t)bins * K * 2 + 16)) return rc;
    if (bits != 0) {
        size_t pb = hp.pbuf_bytes;
        if (int rc = ensure(reinterpret_cast<void**>(&hp.pbuf[0]), &pb, (size_t)(chunk * pitch))) return rc;
        if (int rc = ensure(reinterpret_cast<void**>(&hp.pbuf[1]), &hp.pbuf_bytes, (size_t)(chunk * pitch))) return rc;
    }
    if (scores_host != nullptr) {
        size_t sb = hp.score_bytes;
        if (int rc = ensure(reinterpret_cast<void**>(&hp.scores[0]), &sb, (size_t)chunk * K * 4)) return rc;
        if (int rc = ensure(reinterpret_cast<void**>(&hp.scores[1]), &hp.score_bytes, (size_t)chunk * K * 4)) return rc;
    }
    int64_t* n_dev = hp.tables;
    float* e_dev = reinterpret_cast<float*>(hp.tables + EPI_MAX_STATES * EPI_MAX_STATES);

    // ---- pass 1: stream the matrix in, count ----
    for (int64_t c = 0; c < nchunks; ++c) {
        const int b = (int)(c & 1);
        const int64_t lo = c * chunk;
        const int64_t nb = (bins - lo) < chunk ? (bins - lo) : chunk;
        if (c >= 2) EPI_CUDA(cudaStreamWaitEvent(hp.copy, hp.counted[b], 0));
        if (bits != 0)         // packed rows: one contiguous DMA of 4 / 5 bits per label
            EPI_CUDA(cudaMemcpyAsync(hp.pbuf[b], x_host + lo * pitch, (size_t)(nb * pitch), cudaMemcpyHostToDevice, hp.copy));
        else if (pitch == dpitch)   // already in the device layout: one contiguous DMA (pad bytes travel, never read)
            EPI_CUDA(cudaMemcpyAsync(hp.xbuf[b], x_host + lo * pitch, (size_t)(nb * pitch), cudaMemcpyHostToDevice,
                                     hp.copy));
        else
            EPI_CUDA(cudaMemcpy2DAsync(hp.xbuf[b], (size_t)dpitch, x_host + lo * pitch, (size_t)pitch, (size_t)cols,
                                       (size_t)nb, cudaMemcpyHostToDevice, hp.copy));
        EPI_CUDA(cudaEventRecord(hp.copied[b], hp.copy));
        EPI_CUDA(cudaStreamWaitEvent(hp.compute, hp.copied[b], 0));
        if (bits != 0)
            if (int rc = epi_unpack_states(hp.pbuf[b], nb, cols, bits, pitch, hp.xbuf[b], dpitch, hp.compute)) return rc;
        if (int rc = epi_bin_counts(hp.xbuf[b], nb, cols, dpitch, K, hp.cnt + lo * K, hp.compute)) return rc;
        EPI_CUDA(cudaEventRecord(hp.counted[b], hp.compute));
    }
    // ---- expected table ----
    EPI_CUDA(cudaMemsetAsync(n_dev, 0, (size_t)ntab * 8, hp.compute));
    if (int rc = epi_expected_s1s2(hp.cnt, bins, K, cols, saliency == 1 ? n_dev : nullptr,
                                   saliency == 2 ? n_dev : nullptr, hp.compute))
        return rc;
    if (int rc = epi_normalize_i64(n_dev, ntab, e_dev, hp.compute)) return rc;
    if (counts_host)
        EPI_CUDA(cudaMemcpyAsync(counts_host, n_dev, (size_t)ntab * 8, cudaMemcpyDeviceToHost, hp.compute));
    if (exp_host) EPI_CUDA(cudaMemcpyAsync(exp_host, e_dev, (size_t)ntab * 4, cudaMemcpyDeviceToHost, hp.compute));
    // ---- pass 2: scores, D2H overlapped ----
    if (scores_host != nullptr) {
        for (int64_t c = 0; c < nchunks; ++c) {
            const int b = (int)(c & 1);
            const int64_t lo = c * chunk;
            const int64_t nb = (bins - lo) < chunk ? (bins - lo) : chunk;
            if (c >= 2) EPI_CUDA(cudaStreamWaitEvent(hp.compute, hp.d2h_done[b], 0));
            int rc;
            if (saliency == 1)
                rc = epi_scores_s1(hp.cnt + lo * K, nb, K, cols, e_dev, hp.scores[b], nullptr, EPI_SCORE_TABLE, hp.compute);
            else
                rc = epi_scores_s2(hp.cnt + lo * K, nb, K, cols, (int64_t)cols * (cols - 1), e_dev, hp.scores[b],
                                   nullptr, EPI_SCORE_TABLE, hp.compute);
            if (rc) return rc;
            EPI_CUDA(cudaEventRecord(hp.scored[b], hp.compute));
            EPI_CUDA(cudaStreamWaitEvent(hp.d2h, hp.scored[b], 0));
            EPI_CUDA(cudaMemcpyAsync(scores_host + lo * K, hp.scores[b], (size_t)nb * K * 4, cudaMemcpyDeviceToHost,
                                     hp.d2h));
            EPI_CUDA(cudaEventRecord(hp.d2h_done[b], hp.d2h));
        }
    }
    EPI_CUDA(cudaStreamSynchronize(hp.compute));
    EPI_CUDA(cudaStreamSynchronize(hp.copy));
    EPI_CUDA(cudaStreamSynchronize(hp.d2h));
    return 0;
}

extern "C" int epi_single_host(const int8_t* x_host, int64_t bins, int32_t cols, int64_t pitch, int32_t K,
                               int32_t saliency, int64_t* counts_host, float* exp_host, float* scores_host) {
    return single_host_impl(reinterpret_cast<const uint8_t*>(x_host), bins, cols, pitch, 0, K, saliency, counts_host,
                            exp_host, scores_host);
}

extern "C" int epi_single_host_packed(const uint8_t* packed_host, int64_t bins, int32_t cols, int64_t packed_pitch,
                                      int32_t bits, int32_t K, int32_t saliency, int64_t* counts_host, float* exp_host,
                                      float* scores_host) {
    EPI_REQUIRE(bits == 4 || bits == 5, "bits=%d: the packed layout holds 4 or 5 bits per label", bits);
    return single_host_impl(packed_host, bins, cols, packed_pitch, bits, K, saliency, counts_host, exp_host, scores_host);
}

// ================================================================================================
// S3 and paired mode with HOST buffers: the same stage sequence the Python drivers run (expected.py / scores.py mirrors),
// composed from the device-level entry points, for callers that hold their matrices in host memory.
// ================================================================================================
namespace epi {

struct DevBuf {          // stream-ordered device allocation, freed on scope exit
    void* p = nullptr;
    cudaStream_t st;
    explicit DevBuf(cudaStream_t s) : st(s) {}
    ~DevBuf() {
        if (p) cudaFreeAsync(p, st);
    }
    int alloc(size_t bytes) {
        EPI_CUDA(cudaMallocAsync(&p, bytes ? bytes : 16, st));
        return 0;
    }
    template <class T>
    T* as() const {
        return static_cast<T*>(p);
    }
};

static int upload_matrix(const int8_t* x_host, int64_t bins, int32_t cols, int64_t pitch, int8_t* x_dev, int64_t dpitch,
                         cudaStream_t st) {
    if (pitch == dpitch)
        EPI_CUDA(cudaMemcpyAsync(x_dev, x_host, (size_t)(bins * pitch), cudaMemcpyHostToDevice, st));
    else
        EPI_CUDA(cudaMemcpy2DAsync(x_dev, (size_t)dpitch, x_host, (size_t)pitch, (size_t)cols, (size_t)bins,
                                   cudaMemcpyHostToDevice, st));
    return 0;
}

__global__ void add_counts_kernel(const uint16_t* __restrict__ a, const uint16_t* __restrict__ b, long long n,
                                  uint16_t* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = (uint16_t)(a[i] + b[i]);
}

}  // namespace epi

// expected.main (S3) -> expectedCombination.main -> scores.main (S3) for one in-memory matrix (expected.py:165-204,
// expectedCombination.py:42, scores.py:455-506).  exp_host: float32 [C][C][K][K] or NULL; scores_host: float32 [bins][K].
extern "C" int epi_s3_host(const int8_t* x_host, int64_t bins, int32_t cols, int64_t pitch, int32_t K, float* exp_host,
                           float* scores_host) {
    if (check_device()) return 3;
    EPI_REQUIRE(bins >= 1 && bins < (1ll << 31) && cols >= 2 && cols <= 65535 && pitch >= cols, "bad S3 shape");
    EPI_REQUIRE(K >= 1 && K <= EPI_MAX_STATES, "num_states=%d out of range [1, %d]", K, EPI_MAX_STATES);
    EPI_REQUIRE(x_host != nullptr, "null matrix pointer");
    std::lock_guard<std::mutex> lock(g_pipe_mutex);
    HostPipe& hp = g_pipe;
    if (int rc = pipe_init(hp)) return rc;
    cudaStream_t st = hp.compute;
    const int64_t dpitch = ((int64_t)cols + 15) & ~15ll;
    const int64_t chunk_bins = 131072;                       // bins per Gram launch (see engine.S3_CHUNK_BINS)
    int64_t mp = 0, bp = 0, ntiles = 0, oh_bytes = 0, tile_bytes = 0;
    if (int rc = epi_s3_plan(bins < chunk_bins ? bins : chunk_bins, cols, K, &mp, &bp, &ntiles, &oh_bytes, &tile_bytes)) return rc;
    DevBuf x(st), oht(st), tiles(st), exp3(st), terms(st), scores(st);
    if (int rc = x.alloc((size_t)(bins * dpitch))) return rc;
    if (int rc = oht.alloc((size_t)oh_bytes)) return rc;
    if (int rc = tiles.alloc((size_t)tile_bytes)) return rc;
    const size_t n4 = (size_t)cols * cols * K * K;
    if (int rc = exp3.alloc(n4 * 4)) return rc;
    if (int rc = upload_matrix(x_host, bins, cols, pitch, x.as<int8_t>(), dpitch, st)) return rc;
    for (int64_t lo = 0; lo < bins; lo += chunk_bins) {
        const int64_t n = (bins - lo) < chunk_bins ? (bins - lo) : chunk_bins;
        const int64_t bpc = (n + 127) / 128 * 128;
        if (int rc = epi_s3_onehot(x.as<int8_t>() + lo * dpitch, n, cols, dpitch, K, oht.as<int8_t>(), mp, bpc, st)) return rc;
        if (int rc = epi_s3_gram(oht.as<int8_t>(), mp, bpc, tiles.as<int32_t>(), lo ? 1 : 0, st)) return rc;
    }
    if (int rc = epi_s3_finalize(tiles.as<int32_t>(), cols, K, mp, bins, nullptr, exp3.as<float>(), st)) return rc;
    if (exp_host) EPI_CUDA(cudaMemcpyAsync(exp_host, exp3.p, n4 * 4, cudaMemcpyDeviceToHost, st));
    if (scores_host) {
        int64_t nterms = 0;
        if (int rc = epi_s3_terms_size(cols, K, &nterms)) return rc;
        if (int rc = terms.alloc((size_t)nterms * 8)) return rc;
        if (int rc = scores.alloc((size_t)bins * K * 4)) return rc;
        if (int rc = epi_s3_terms(exp3.as<float>(), cols, K, terms.as<double>(), st)) return rc;
        if (int rc = epi_scores_s3(x.as<int8_t>(), bins, cols, dpitch, K, terms.as<double>(), scores.as<float>(), nullptr, st))
            return rc;
        EPI_CUDA(cudaMemcpyAsync(scores_host, scores.p, (size_t)bins * K * 4, cudaMemcpyDeviceToHost, st));
    }
    EPI_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// Paired mode for one pair of in-memory matrices: expected table of the union [A | B] (helpers.py:173-179), scores of both
// groups, delta, quiescence mask, and `nperm` device-drawn null shuffles per bin with their signed squared distances
// (scores.py:172-256; the reference draws one shuffle).  saliency 1 or 2; group_size -1 = the groups' own widths (-g
// otherwise, clipped like the reference's slices); bin_offset = global index of row 0 (keys the random streams).
// Outputs (any may be NULL): counts_host int64 [K] or [K][K], exp_host float32 same shape, delta_host float32 [bins][K],
// null_host float32 [nperm][bins], quiescent_host uint8 [bins].
extern "C" int epi_paired_host(const int8_t* xa_host, int64_t pitch_a, int32_t cols_a, const int8_t* xb_host,
                               int64_t pitch_b, int32_t cols_b, int64_t bins, int32_t K, int32_t saliency,
                               int32_t quiescent_state, int32_t group_size, uint64_t seed, int64_t bin_offset,
                               int32_t nperm, int64_t* counts_host, float* exp_host, float* delta_host, float* null_host,
                               uint8_t* quiescent_host) {
    if (check_device()) return 3;
    EPI_REQUIRE(saliency == 1 || saliency == 2, "Please ensure that saliency metric is either 1 or 2 for Pairwise Epilogos");
    EPI_REQUIRE(bins >= 1 && bins < (1ll << 31) && cols_a >= 2 && cols_b >= 2 && pitch_a >= cols_a && pitch_b >= cols_b,
                "bad paired shape");
    EPI_REQUIRE(K >= 1 && K <= EPI_MAX_STATES && nperm >= 0, "bad paired arguments");
    EPI_REQUIRE(xa_host != nullptr && xb_host != nullptr, "null matrix pointer");
    std::lock_guard<std::mutex> lock(g_pipe_mutex);
    HostPipe& hp = g_pipe;
    if (int rc = pipe_init(hp)) return rc;
    cudaStream_t st = hp.compute;
    const int n = cols_a + cols_b;
    const int size_a = group_size < 0 ? cols_a : (group_size < n ? group_size : n);
    int size_b = group_size < 0 ? cols_b : (n - group_size < group_size ? n - group_size : group_size);
    if (size_b < 0) size_b = 0;
    const int64_t pa = ((int64_t)cols_a + 15) & ~15ll, pb = ((int64_t)cols_b + 15) & ~15ll;
    const int ntab = saliency == 1 ? K : K * K;
    const int64_t p1 = (int64_t)cols_a * (cols_a - 1), p2 = (int64_t)cols_b * (cols_b - 1);
    DevBuf xa(st), xb(st), ca(st), cb(st), cc(st), sa(st), sb(st), delta(st), mask(st), oa(st), ob(st), na(st), nb(st), nd(st);
    if (int rc = xa.alloc((size_t)(bins * pa))) return rc;
    if (int rc = xb.alloc((size_t)(bins * pb))) return rc;
    if (int rc = ca.alloc((size_t)bins * K * 2)) return rc;
    if (int rc = cb.alloc((size_t)bins * K * 2)) return rc;
    if (int rc = cc.alloc((size_t)bins * K * 2)) return rc;
    if (int rc = upload_matrix(xa_host, bins, cols_a, pitch_a, xa.as<int8_t>(), pa, st)) return rc;
    if (int rc = upload_matrix(xb_host, bins, cols_b, pitch_b, xb.as<int8_t>(), pb, st)) return rc;
    if (int rc = epi_bin_counts(xa.as<int8_t>(), bins, cols_a, pa, K, ca.as<uint16_t>(), st)) return rc;
    if (int rc = epi_bin_counts(xb.as<int8_t>(), bins, cols_b, pb, K, cb.as<uint16_t>(), st)) return rc;
    add_counts_kernel<<<persistent_grid((bins * K + 255) / 256, 8), 256, 0, st>>>(ca.as<uint16_t>(), cb.as<uint16_t>(),
                                                                                 (long long)bins * K, cc.as<uint16_t>());
    EPI_CUDA(cudaGetLastError());
    int64_t* n_dev = hp.tables;
    float* e_dev = reinterpret_cast<float*>(hp.tables + EPI_MAX_STATES * EPI_MAX_STATES);
    EPI_CUDA(cudaMemsetAsync(n_dev, 0, (size_t)ntab * 8, st));
    if (int rc = epi_expected_s1s2(cc.as<uint16_t>(), bins, K, n, saliency == 1 ? n_dev : nullptr,
                                   saliency == 2 ? n_dev : nullptr, st))
        return rc;
    if (int rc = epi_normalize_i64(n_dev, ntab, e_dev, st)) return rc;
    if (counts_host) EPI_CUDA(cudaMemcpyAsync(counts_host, n_dev, (size_t)ntab * 8, cudaMemcpyDeviceToHost, st));
    if (exp_host) EPI_CUDA(cudaMemcpyAsync(exp_host, e_dev, (size_t)ntab * 4, cudaMemcpyDeviceToHost, st));
    auto score = [&](const uint16_t* c, int64_t rows, int width, int64_t perms, float* out) -> int {
        if (saliency == 1) return epi_scores_s1(c, rows, K, width > 0 ? width : 1, e_dev, out, nullptr, EPI_SCORE_TABLE, st);
        return epi_scores_s2(c, rows, K, width > 0 ? width : 1, perms, e_dev, out, nullptr, EPI_SCORE_TABLE, st);
    };
    if (delta_host) {
        if (int rc = sa.alloc((size_t)bins * K * 4)) return rc;
        if (int rc = sb.alloc((size_t)bins * K * 4)) return rc;
        if (int rc = delta.alloc((size_t)bins * K * 4)) return rc;
        if (int rc = score(ca.as<uint16_t>(), bins, cols_a, p1, sa.as<float>())) return rc;
        if (int rc = score(cb.as<uint16_t>(), bins, cols_b, p2, sb.as<float>())) return rc;
        if (int rc = epi_pairwise_combine(sa.as<float>(), sb.as<float>(), nullptr, nullptr, bins, K, delta.as<float>(), nullptr, st))
            return rc;
        EPI_CUDA(cudaMemcpyAsync(delta_host, delta.p, (size_t)bins * K * 4, cudaMemcpyDeviceToHost, st));
    }
    if (quiescent_host) {
        if (int rc = mask.alloc((size_t)bins)) return rc;
        if (int rc = epi_quiescent_mask(ca.as<uint16_t>(), cb.as<uint16_t>(), bins, K, cols_a, cols_b, quiescent_state,
                                        mask.as<uint8_t>(), st))
            return rc;
        EPI_CUDA(cudaMemcpyAsync(quiescent_host, mask.p, (size_t)bins, cudaMemcpyDeviceToHost, st));
    }
    if (null_host && nperm > 0) {
        int batch = (int)((int64_t)(256ll << 20) / (bins * K * 4));        // ~256 MB of null scores per group at a time
        if (batch < 1) batch = 1;
        if (batch > nperm) batch = nperm;
        if (int rc = oa.alloc((size_t)batch * bins * K * 2)) return rc;
        if (int rc = ob.alloc((size_t)batch * bins * K * 2)) return rc;
        if (int rc = na.alloc((size_t)batch * bins * K * 4)) return rc;
        if (int rc = nb.alloc((size_t)batch * bins * K * 4)) return rc;
        if (int rc = nd.alloc((size_t)nperm * bins * 4)) return rc;
        // the philox counter carries the permutation index: batch [done, done + nbatch) draws permutations done .. done +
        // nbatch - 1 of the one (seed, global bin) stream, so null row p does not depend on the batch size (nor on bins)
        for (int done = 0; done < nperm; done += batch) {
            const int nbatch = (nperm - done) < batch ? (nperm - done) : batch;
            if (int rc = epi_shuffled_counts_philox_range(ca.as<uint16_t>(), cb.as<uint16_t>(), bins, K, n, size_a, size_b,
                                                          seed, bin_offset, done, nbatch, oa.as<uint16_t>(),
                                                          ob.as<uint16_t>(), st))
                return rc;
            if (int rc = score(oa.as<uint16_t>(), (int64_t)nbatch * bins, size_a, p1, na.as<float>())) return rc;
            if (int rc = score(ob.as<uint16_t>(), (int64_t)nbatch * bins, size_b, p2, nb.as<float>())) return rc;
            if (int rc = epi_pairwise_combine(nullptr, nullptr, na.as<float>(), nb.as<float>(), (int64_t)nbatch * bins, K,
                                              nullptr, nd.as<float>() + (int64_t)done * bins, st))
                return rc;
        }
        EPI_CUDA(cudaMemcpyAsync(null_host, nd.p, (size_t)nperm * bins * 4, cudaMemcpyDeviceToHost, st));
    }
    EPI_CUDA(cudaStreamSynchronize(st));
    return 0;
}
