// Host-side I/O of the scoring path (SURVEY.md section 8f, row f3): the callers and data formats either side of
// the kernels.  Pure host code (compiled by nvcc for convenience, links zlib).
//
//   epi_tsv_shape        rows (newline count, helpers.countRows helpers.py:80-99) and columns of the first line
//   epi_pack_tsv         rows [lo, hi) of `chr start end s_1 .. s_C` -> int8 labels-1 in the kernels' pitched
//                        layout + start/end/chromosome per row (replaces the pandas parse of helpers.readStates,
//                        helpers.py:150-168, and of scores.py:161); labels are validated here
//   epi_scores_tsv_*     score text back into float64 rows (similaritySearch_max_mean.readScores, :51-74)
//   epi_write_scores_gz  `chr \t start \t end \t K x "%.5f"` lines through gzip (scores.writeScores,
//                        scores.py:509-536): rows are formatted and deflated in parallel as independent gzip
//                        members (a valid multi-member .gz; the decompressed text is byte-identical to the
//                        reference's)
#include <math.h>
#include <sched.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>

#include <algorithm>
#include <memory>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "common.cuh"
#include "fast_inflate.h"
#include "label_simd.h"
#include "parallel_inflate.h"

namespace epi {

// Thread budget of one reader.  Every file being read has an inflate stage and a parse stage; several files may be read
// at once (session.prefetch) and, under torchrun, several ranks share the host (LOCAL_WORLD_SIZE), so the machine's
// cores are divided by both before a reader takes its share.
static std::atomic<int> g_active_readers{0};
static std::atomic<int> g_expected_readers{0};      // epi_reader_concurrency: files the caller is about to read at once
static std::atomic<int> g_reading_ranks{0};         // ... and ranks of this host that read at the same time (0: all of them)
static int cores_per_reader() {
    int cores = (int)std::thread::hardware_concurrency();
#ifdef __linux__
    cpu_set_t set;
    CPU_ZERO(&set);
    if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) cores = std::min(cores > 0 ? cores : 1 << 20, CPU_COUNT(&set));
#endif
    if (cores < 1) cores = 1;
    int ranks = 1;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) ranks = std::max(1, atoi(e));
    if (g_reading_ranks.load() > 0) ranks = std::min(ranks, g_reading_ranks.load());
    const int active = std::max(1, std::max(g_active_readers.load(), g_expected_readers.load()));
    return std::max(1, cores / (ranks * active));
}
// what the calling thread's last reader did (epi_reader_stats): mode, chunks, chunks with a start, chunks accepted
static thread_local int64_t t_reader_stats[4] = {0, 0, 0, 0};
}  // namespace epi
static int parse_threads();
namespace epi {
// threads that decode ONE gzip stream in parallel (parallel_inflate.h); 1 = the sequential decoder
static int inflate_threads() {
    if (const char* e = getenv("EPI_INFLATE_THREADS")) {
        const int v = atoi(e);
        if (v >= 1) return v > 32 ? 32 : v;
    }
    // three quarters of the reader's cores: decoding, marker resolution and CRC take ~3 ns per byte of text, the SIMD row
    // parser ~1 ns (measured, DESIGN.md)
    const int t = std::min(12, (cores_per_reader() * 3 + 2) / 4);
    return t < 2 ? 1 : t;
}

// "%.5f" of a double with printf semantics (round-half-even on the exact binary value).  Fast path: scale by 1e5 and
// round; whenever the scaled value is within 1e-6 of a rounding boundary (or huge / non-finite) defer to snprintf.
static inline char* format_5f(char* p, double d) {
    if (d != d) return p + sprintf(p, "nan");                    // Python's "{:.5f}" prints nan without a sign; glibc "-nan"
    if (isinf(d)) return p + sprintf(p, d < 0 ? "-inf" : "inf");
    if (!(fabs(d) < 1e9)) return p + sprintf(p, "%.5f", d);
    const bool neg = signbit(d);
    const double a = fabs(d) * 1e5;
    const double fl = floor(a);
    const double frac = a - fl;
    if (fabs(frac - 0.5) < 1e-6) return p + sprintf(p, "%.5f", d);
    unsigned long long q = (unsigned long long)fl + (frac > 0.5 ? 1ull : 0ull);
    if (neg) *p++ = '-';
    const unsigned long long ip = q / 100000ull;
    unsigned fr = (unsigned)(q % 100000ull);
    char tmp[24];
    int n = 0;
    unsigned long long v = ip;
    do {
        tmp[n++] = (char)('0' + v % 10);
        v /= 10;
    } while (v);
    while (n) *p++ = tmp[--n];
    *p++ = '.';
    p[4] = (char)('0' + fr % 10); fr /= 10;
    p[3] = (char)('0' + fr % 10); fr /= 10;
    p[2] = (char)('0' + fr % 10); fr /= 10;
    p[1] = (char)('0' + fr % 10); fr /= 10;
    p[0] = (char)('0' + fr % 10);
    return p + 5;
}

static inline char* format_i64(char* p, long long v) {
    if (v < 0) {
        *p++ = '-';
        v = -v;
    }
    char tmp[24];
    int n = 0;
    do {
        tmp[n++] = (char)('0' + v % 10);
        v /= 10;
    } while (v);
    while (n) *p++ = tmp[--n];
    return p;
}

}  // namespace epi

using namespace epi;

// Line source: a background thread inflates the file into a ring of two large blocks while the caller parses the
// previous one; lines that straddle a block boundary are stitched into a side buffer.  The two threads hand blocks over
// through a mutex + condition variable (no spinning: with one reader per input file running concurrently, a spinning
// parser would take the core its own inflate thread needs).
struct LineSource {
    static constexpr size_t BLOCK = 16u << 20;
    static constexpr size_t HIST = 32768;       // DEFLATE window kept in front of every block for the native decoder
    static constexpr size_t PACK_PAD = 64;      // zero bytes behind the compressed file: the decoders' bit readers run ahead
    gzFile gz = nullptr;
    std::vector<char> blocks[2];                // [HIST bytes of history | BLOCK bytes of text | slack]
    size_t lens[2] = {0, 0};
    std::thread worker;
    std::mutex mu;
    std::condition_variable cv;
    int ready[2] = {0, 0};              // 1 = filled by the worker, 0 = free (guarded by mu)
    bool abort_ = false;                // the reader is going away: stop inflating
    int cur = 0;
    size_t pos = 0;
    std::vector<char> carry;
    std::string path_;
    std::string error_;                 // set by the worker before its last block is published
    std::vector<uint8_t> packed;        // the whole compressed file (native decoder)
    FastInflate inflater;
    ParallelInflate pinflater;          // several threads on the one stream (large files, when cores are free)
    bool native = false;
    bool parallel = false;
    bool counted_ = false;
    uint64_t delivered = 0;             // bytes handed to the parser in complete blocks

    char* text(int w) { return blocks[w].data() + HIST; }

    // the whole file in memory if it is gzip and the native decoder is not disabled (EPI_ZLIB_INFLATE=1)
    bool load_packed(const char* path) {
        if (getenv("EPI_ZLIB_INFLATE") != nullptr) return false;
        FILE* f = fopen(path, "rb");
        if (!f) return false;
        unsigned char magic[2] = {0, 0};
        const bool gzip = fread(magic, 1, 2, f) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
        bool ok = false;
        if (gzip && fseek(f, 0, SEEK_END) == 0) {
            const long long size = ftell(f);
            if (size > 0 && fseek(f, 0, SEEK_SET) == 0) {
                packed.assign((size_t)size + PACK_PAD, 0);
                ok = fread(packed.data(), 1, (size_t)size, f) == (size_t)size;
            }
        }
        fclose(f);
        if (!ok) std::vector<uint8_t>().swap(packed);
        return ok;
    }

    // fill block w with the native decoder; returns the bytes produced (BLOCK unless the stream ended) or -1 on error
    bool after_member_ = false;      // the previous decode call ended exactly at the end of a gzip member
    long long fill_native(int w, uint32_t& crc, uint64_t& member_bytes) {
        uint8_t* base = reinterpret_cast<uint8_t*>(text(w));
        uint8_t* out = base;
        uint8_t* const end = base + BLOCK;
        while (out < end) {
            if (inflater.at_end_of_input()) break;
            uint8_t* np = out;
            const FastInflate::Status st = inflater.decode(out, end, &np);
            crc = crc32_fast(crc, out, (size_t)(np - out));
            member_bytes += (uint64_t)(np - out);
            const bool produced = np != out;
            out = np;
            if (st == FastInflate::ERROR) {
                if (after_member_ && !produced) {
                    // bytes after a complete member that are neither zero padding nor another gzip member: Python's gzip
                    // module (the reference's reader) raises on them; zlib's gzread would silently ignore them
                    error_ = path_ + ": trailing garbage after the last gzip member";
                    return -2;
                }
                return -1;
            }
            after_member_ = false;
            if (st == FastInflate::MEMBER_END) {
                after_member_ = true;
                if (crc != inflater.member_crc() || (uint32_t)member_bytes != inflater.member_isize()) {
                    error_ = path_ + ": gzip member fails its CRC-32 / length check";
                    return -2;
                }
                crc = (uint32_t)crc32(0L, Z_NULL, 0);
                member_bytes = 0;
                if (inflater.only_padding_left()) break;
            }
        }
        return (long long)(out - base);
    }

    // next piece of text from the parallel decoder into block w: bytes, 0 at the end of the stream, -1 = it gave up
    // (the caller falls back to zlib from the bytes already delivered), -2 = error_ is set
    long long fill_parallel(int w) {
        size_t n = 0;
        const int r = pinflater.next(blocks[w], &n);      // swaps the text buffer in; the old one is recycled
        if (r == 1) return (long long)n;
        if (r == 0) return 0;
        if (r == -2) {
            error_ = path_ + ": trailing garbage after the last gzip member";
            return -2;
        }
        return -1;
    }

    bool open(const char* path) {
        path_ = path;
        ++g_active_readers;
        counted_ = true;
        native = load_packed(path);
        if (!native) {
            gz = gzopen(path, "rb");
            if (!gz) return false;
            gzbuffer(gz, 1 << 20);
        } else {
            inflater.reset(packed.data(), packed.size() - PACK_PAD);
            // large single files: decode the one stream with several threads
            const size_t size = packed.size() - PACK_PAD;
            const int threads = inflate_threads();
            size_t chunk = std::min<size_t>(1u << 20, std::max<size_t>(256u << 10, size / (size_t)(8 * std::max(1, threads))));
            size_t least = 2u << 20;
            if (const char* e = getenv("EPI_INFLATE_CHUNK")) {          // test / tuning knob: chunk bytes, no size threshold
                if (atoll(e) > 0) {
                    chunk = (size_t)atoll(e);
                    least = 0;
                }
            }
            // a stream that expands more than ~100-fold (ISIZE of the last member against the file size) would need
            // gigabytes per chunk in flight: such files stay with the sequential decoder and its 16 MB blocks
            const uint64_t isize = size >= 18 ? ((uint64_t)packed[size - 4] | ((uint64_t)packed[size - 3] << 8) |
                                                 ((uint64_t)packed[size - 2] << 16) | ((uint64_t)packed[size - 1] << 24)) : 0;
            const bool dense = isize / 100 <= (uint64_t)size;
            const auto t_s0 = std::chrono::steady_clock::now();
            if (threads >= 2 && size >= least && dense) parallel = pinflater.start(packed.data(), size, threads, chunk, HIST);
            if (getenv("EPI_INFLATE_DEBUG") != nullptr)
                fprintf(stderr, "[epi reader] chunk starts found in %.3f s\n",
                        std::chrono::duration<double>(std::chrono::steady_clock::now() - t_s0).count());
        }
        blocks[0].resize(HIST + BLOCK + 64);
        blocks[1].resize(HIST + BLOCK + 64);
        worker = std::thread([this]() {
            int w = 0;
            uint32_t crc = (uint32_t)crc32(0L, Z_NULL, 0);
            uint64_t member_bytes = 0;
            for (;;) {
                {
                    std::unique_lock<std::mutex> lk(mu);
                    cv.wait(lk, [&] { return ready[w] == 0 || abort_; });
                    if (abort_) return;
                }
                long long n;
                if (!parallel && blocks[w].size() < HIST + BLOCK + 64) blocks[w].resize(HIST + BLOCK + 64);   // after a parallel piece
                if (native) {
                    std::string why;
                    if (parallel) {
                        n = fill_parallel(w);
                        if (n == -1) {
                            {
                                std::lock_guard<std::mutex> lk(mu);
                                if (abort_) return;              // the reader is going away, not a decoding failure
                            }
                            why = pinflater.error();
                            pinflater.stop();
                            parallel = false;
                            if (blocks[w].size() < HIST + BLOCK + 64) blocks[w].resize(HIST + BLOCK + 64);
                        }
                    } else {
                        // the last 32 KiB of the previous block are the window of the next one
                        if (delivered) memcpy(blocks[w].data(), text(w ^ 1) + BLOCK - HIST, HIST);
                        n = fill_native(w, crc, member_bytes);
                        if (n == -1) why = inflater.error();
                    }
                    if (n == -1) {
                        // The native decoder gave up (a stream it does not understand): hand the file to zlib, skip
                        // what the parser already has, and carry on from there.  Corrupt data fails in zlib as well.
                        native = false;
                        gz = gzopen(path_.c_str(), "rb");
                        n = -3;
                        if (gz) {
                            gzbuffer(gz, 1 << 20);
                            uint64_t skip = delivered;
                            bool ok = true;
                            while (skip && ok) {
                                const unsigned chunk = (unsigned)std::min<uint64_t>(skip, BLOCK);
                                ok = gzread(gz, text(w), chunk) == (int)chunk;
                                skip -= chunk;
                            }
                            if (ok) n = gzread(gz, text(w), (unsigned)BLOCK);
                        }
                        if (n < 0) error_ = path_ + ": cannot inflate (" + why + ")";
                    }
                } else {
                    n = gzread(gz, text(w), (unsigned)BLOCK);
                }
                if (!native && gz != nullptr && n < (long long)BLOCK && error_.empty()) {
                    // end of file or failure: zlib reports a stream cut short (Z_BUF_ERROR) or corrupt data only here
                    int errnum = Z_OK;
                    const char* msg = gzerror(gz, &errnum);
                    if (n < 0 || (errnum != Z_OK && errnum != Z_STREAM_END))
                        error_ = path_ + ": " + (msg && *msg ? msg : "gzip stream is damaged or cut short");
                }
                const bool last = n <= 0 || (native && !parallel && (size_t)n < BLOCK);
                {
                    std::lock_guard<std::mutex> lk(mu);
                    lens[w] = n > 0 ? (size_t)n : 0;
                    ready[w] = 1;
                }
                cv.notify_all();
                if (n > 0) delivered += (uint64_t)n;
                if (last && n <= 0) return;
                if (last) {
                    // a short native block is the end of the stream: publish the empty block that marks it
                    w ^= 1;
                    std::unique_lock<std::mutex> lk(mu);
                    cv.wait(lk, [&] { return ready[w] == 0 || abort_; });
                    if (abort_) return;
                    lens[w] = 0;
                    ready[w] = 1;
                    lk.unlock();
                    cv.notify_all();
                    return;
                }
                w ^= 1;
            }
        });
        wait_filled(0);
        return true;
    }
    // empty unless inflating failed; valid once next_line() has returned false
    const std::string& error() {
        std::lock_guard<std::mutex> lk(mu);
        return error_;
    }
    void wait_filled(int b) {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return ready[b] == 1; });
    }
    // advance to the next block; false at end of file
    bool next_block() {
        if (lens[cur] == 0) return false;          // the empty block marks the end of the stream: nothing follows it
        {
            std::lock_guard<std::mutex> lk(mu);
            ready[cur] = 0;
        }
        cv.notify_all();
        cur ^= 1;
        wait_filled(cur);
        pos = 0;
        return lens[cur] != 0;
    }
    // the unread rest of the current block, then the following blocks (raw byte stream; do not mix with next_line)
    bool next_raw(const char*& b, size_t& n) {
        if (pos >= lens[cur] && !next_block()) return false;
        b = text(cur) + pos;
        n = lens[cur] - pos;
        pos = lens[cur];
        return n != 0;
    }
    // next line [begin, end) without the newline; returns false at end of file.  has_nl tells whether the line was
    // terminated (the reference counts newline characters, helpers.py:92-97).
    bool next_line(const char*& begin, const char*& end, bool& has_nl) {
        for (;;) {
            const char* base = text(cur);
            const size_t len = lens[cur];
            if (pos < len) {
                const char* nl = static_cast<const char*>(memchr(base + pos, '\n', len - pos));
                if (nl != nullptr && carry.empty()) {
                    begin = base + pos;
                    end = nl;
                    pos = (size_t)(nl - base) + 1;
                    has_nl = true;
                    return true;
                }
                if (nl != nullptr) {
                    carry.insert(carry.end(), base + pos, nl);
                    pos = (size_t)(nl - base) + 1;
                    line_buf.swap(carry);
                    carry.clear();
                    begin = line_buf.data();
                    end = line_buf.data() + line_buf.size();
                    has_nl = true;
                    return true;
                }
                carry.insert(carry.end(), base + pos, base + len);
                pos = len;
            }
            if (!next_block()) {
                if (carry.empty()) return false;
                line_buf.swap(carry);
                carry.clear();
                begin = line_buf.data();
                end = line_buf.data() + line_buf.size();
                has_nl = false;
                return true;
            }
        }
    }
    std::vector<char> line_buf;

    // Every complete line that can be handed out without letting go of the current block (the first one may be the line
    // that straddled the previous block boundary; it lives in line_buf).  The pointers stay valid until the next call.
    // Returns false at end of file; an unterminated tail at the end of the file is not a line (countRows semantics) and
    // is dropped.  Do not mix with next_line().
    bool next_batch(std::vector<std::pair<const char*, const char*>>& lines) {
        lines.clear();
        for (;;) {
            const char* base = text(cur);
            const size_t len = lens[cur];
            while (pos < len) {
                const char* nl = static_cast<const char*>(memchr(base + pos, '\n', len - pos));
                if (nl == nullptr) break;
                if (!carry.empty()) {
                    carry.insert(carry.end(), base + pos, nl);
                    line_buf.swap(carry);
                    carry.clear();
                    lines.emplace_back(line_buf.data(), line_buf.data() + line_buf.size());
                } else {
                    lines.emplace_back(base + pos, nl);
                }
                pos = (size_t)(nl - base) + 1;
            }
            if (!lines.empty()) return true;           // the partial tail is picked up by the next call
            if (pos < len) {
                carry.insert(carry.end(), base + pos, base + len);
                pos = len;
            }
            if (!next_block()) return false;
        }
    }
    ~LineSource() {
        if (worker.joinable()) {
            {
                std::lock_guard<std::mutex> lk(mu);
                abort_ = true;
            }
            cv.notify_all();
            pinflater.stop();              // a worker blocked in the parallel decoder's next() wakes up with a failure
            worker.join();
        }
        if (gz) gzclose(gz);
        if (counted_) --g_active_readers;
        size_t c = 0, f = 0, a = 0;
        pinflater.stats(&c, &f, &a);
        t_reader_stats[0] = c ? (parallel ? 2 : 3) : (native ? 1 : 0);
        t_reader_stats[1] = (int64_t)c;
        t_reader_stats[2] = (int64_t)f;
        t_reader_stats[3] = (int64_t)a;
        if (getenv("EPI_INFLATE_DEBUG") != nullptr) {
            fprintf(stderr, "[epi reader] %s: %s, %zu chunks, %zu with a start, %zu accepted, %llu bytes delivered\n", path_.c_str(),
                    c ? (parallel ? "parallel inflate" : "parallel inflate abandoned") : (native ? "sequential inflate" : "zlib"), c, f, a,
                    (unsigned long long)delivered);
            if (c)
                fprintf(stderr, "[epi reader]   pool time: decode %.3f s, waiting for the predecessor %.3f s, resolve + CRC-32 %.3f s\n",
                        pinflater.us_decode.load() * 1e-6, pinflater.us_wait.load() * 1e-6, pinflater.us_resolve.load() * 1e-6);
        }
    }
};

extern "C" int epi_tsv_shape(const char* path, int64_t* rows_out, int32_t* cols_out) {
    EPI_REQUIRE(path != nullptr, "null path");
    LineSource src;                                       // the library's decoders (several threads on a large file)
    EPI_REQUIRE(src.open(path), "cannot open %s", path);
    int64_t rows = 0;
    int32_t tabs_first = 0;
    bool first = true;
    const char* b;
    size_t n;
    while (src.next_raw(b, n)) {
        size_t i = 0;
        if (first) {
            for (; i < n; ++i) {
                if (b[i] == '\t') ++tabs_first;
                else if (b[i] == '\n') {
                    first = false;
                    break;
                }
            }
        }
        const char* p = b + i;
        const char* const e = b + n;
        while (p < e) {                                   // newline count as in helpers.countRows (helpers.py:92-97)
            const char* q = static_cast<const char*>(memchr(p, '\n', (size_t)(e - p)));
            if (q == nullptr) break;
            ++rows;
            p = q + 1;
        }
    }
    EPI_REQUIRE(src.error().empty(), "%s", src.error().c_str());
    if (rows_out) *rows_out = rows;
    if (cols_out) *cols_out = tabs_first + 1 - 3;           // biosample columns (after chr, start, end)
    return 0;
}

// One row `chr \t start \t end \t s_1 .. s_C` -> labels-1 in dst[0..cols), coordinates, chromosome id (names grows).
// Returns 0, or 2 with the error set.
static int parse_row(const char* path, int64_t row, const char* p, const char* e, int32_t cols, int32_t num_states,
                     int8_t* dst, int64_t* start, int64_t* end, int32_t* chrom, std::vector<std::string>& names,
                     int& last_id, bool want_chrom) {
    if (e > p && e[-1] == '\r') --e;
    // ---- chromosome name ----
    const char* t = static_cast<const char*>(memchr(p, '\t', (size_t)(e - p)));
    EPI_REQUIRE(t != nullptr, "%s: row %lld is truncated (expected chr<TAB>start<TAB>end<TAB>states)", path,
                (long long)row);
    if (want_chrom) {
        const size_t nl = (size_t)(t - p);
        int id = -1;
        if (last_id >= 0 && names[last_id].size() == nl && memcmp(names[last_id].data(), p, nl) == 0) id = last_id;
        for (size_t i = 0; id < 0 && i < names.size(); ++i)
            if (names[i].size() == nl && memcmp(names[i].data(), p, nl) == 0) id = (int)i;
        if (id < 0) {
            id = (int)names.size();
            names.emplace_back(p, nl);
        }
        *chrom = last_id = id;
    }
    p = t + 1;
    // ---- start, end ----
    for (int f = 0; f < 2; ++f) {
        long long v = 0;
        bool negv = false;
        if (p < e && *p == '-') {
            negv = true;
            ++p;
        }
        const char* d0 = p;
        while (p < e && *p >= '0' && *p <= '9') v = v * 10 + (*p++ - '0');
        EPI_REQUIRE(p > d0 && p < e && *p == '\t', "%s: row %lld: bad coordinate field", path, (long long)row);
        ++p;
        if (f == 0 && start) *start = negv ? -v : v;
        if (f == 1 && end) *end = negv ? -v : v;
    }
    // ---- state labels: 1..num_states, one to three digits ----
    int j = 0;
    // wide rows: 16 bytes at a time (label_simd.cpp) up to the last few labels; anything but one- and two-digit labels in
    // range makes it step back (-1) and the scalar loops below parse the row from here and report what is wrong
    if (cols >= 48 && label_simd_available() && getenv("EPI_PARSE_SCALAR") == nullptr) {      // (the knob: for A/B runs and tests)
        const char* resume = p;
        const int got = parse_labels_simd(p, e, cols - 1, num_states, dst, &resume);
        if (got > 0) {
            j = got;
            p = resume;
        }
    }
    // fast path for all but the last column: a one- or two-digit label and its tab, three comparisons per label.  Anything
    // else (three digits, a bad character, a label out of range, a short row) falls through to the careful loop below,
    // which parses it again from the same position and reports what is wrong.
    while (j + 1 < cols && e - p >= 4) {
        // (measured alternatives: a branch-free selection between the two shapes is 40 % slower, an AVX2 tab-mask walk
        // 15 % slower on realistic matrices -- with branches the predictor follows the dominant label and speculation
        // hides the load-to-advance dependency; only matrices with unpredictable label widths would gain from SIMD)
        const unsigned d0 = (unsigned)(p[0] - '0'), d1 = (unsigned)(p[1] - '0');
        unsigned v, adv;
        if (p[1] == '\t') {
            v = d0;
            adv = 2;
        } else if (p[2] == '\t' && d1 <= 9u) {
            v = d0 * 10u + d1;
            adv = 3;
        } else {
            break;
        }
        if (d0 > 9u || v - 1u >= (unsigned)num_states) break;
        dst[j++] = (int8_t)(v - 1u);
        p += adv;
    }
    while (j < cols) {
        EPI_REQUIRE(p < e, "%s: row %lld has %d state columns, expected %d", path, (long long)row, j, cols);
        unsigned v = (unsigned)(*p - '0');
        EPI_REQUIRE(v <= 9, "%s: row %lld column %d: state label is not an integer", path, (long long)row, j + 4);
        ++p;
        while (p < e && (unsigned)(*p - '0') <= 9) {
            v = v * 10 + (unsigned)(*p++ - '0');
            EPI_REQUIRE(v <= 1000, "%s: row %lld column %d: state label out of range", path, (long long)row, j + 4);
        }
        EPI_REQUIRE(v >= 1 && v <= (unsigned)num_states, "%s: row %lld column %d: state %u outside 1..%d", path,
                    (long long)row, j + 4, v, num_states);
        dst[j++] = (int8_t)(v - 1);
        if (p < e) {
            EPI_REQUIRE(*p == '\t', "%s: row %lld column %d: unexpected character", path, (long long)row, j + 3);
            ++p;
            EPI_REQUIRE(j < cols || p == e, "%s: row %lld has more than %d state columns", path, (long long)row, cols);
        }
    }
    EPI_REQUIRE(p == e, "%s: row %lld has more than %d state columns", path, (long long)row, cols);
    return 0;
}

static int emit_names(const std::vector<std::string>& names, char* chrom_names, int32_t chrom_names_cap) {
    if (chrom_names == nullptr) return 0;
    size_t off = 0;
    for (const std::string& s : names) {
        EPI_REQUIRE(off + s.size() + 1 <= (size_t)chrom_names_cap, "chromosome name buffer too small");
        memcpy(chrom_names + off, s.c_str(), s.size() + 1);
        off += s.size() + 1;
    }
    return 0;
}

// The reader's decompressed byte stream of a file (what the parsers see): a diagnostic / test entry for the native
// DEFLATE decoder.  Copies at most cap bytes into out (may be NULL) and returns the stream's total length in *n_out.
extern "C" int epi_inflate_file(const char* path, uint8_t* out, int64_t cap, int64_t* n_out) {
    EPI_REQUIRE(path != nullptr && n_out != nullptr, "null pointer argument");
    LineSource src;
    EPI_REQUIRE(src.open(path), "cannot open %s", path);
    int64_t total = 0;
    const char* b;
    size_t n;
    while (src.next_raw(b, n)) {
        if (out != nullptr && total < cap) memcpy(out + total, b, (size_t)std::min<int64_t>((int64_t)n, cap - total));
        total += (int64_t)n;
    }
    EPI_REQUIRE(src.error().empty(), "%s", src.error().c_str());
    *n_out = total;
    return 0;
}

extern "C" int epi_reader_concurrency(int32_t files, int32_t ranks) {
    g_expected_readers.store(files > 0 ? files : 0);
    g_reading_ranks.store(ranks > 0 ? ranks : 0);
    return 0;
}

extern "C" int epi_reader_threads(int32_t* inflate_out, int32_t* parse_out) {
    if (inflate_out) *inflate_out = inflate_threads();
    if (parse_out) *parse_out = parse_threads();
    return 0;
}

extern "C" int epi_reader_stats(int64_t* out4) {
    EPI_REQUIRE(out4 != nullptr, "null pointer argument");
    for (int i = 0; i < 4; ++i) out4[i] = t_reader_stats[i];
    return 0;
}

extern "C" int epi_pack_tsv(const char* path, int64_t row_lo, int64_t row_hi, int32_t cols, int32_t num_states,
                            int8_t* out, int64_t pitch, int64_t* starts, int64_t* ends, int32_t* chrom_id,
                            char* chrom_names, int32_t chrom_names_cap, int32_t* n_chrom_out) {
    EPI_REQUIRE(path != nullptr && (out != nullptr || row_hi == row_lo), "null pointer argument");
    EPI_REQUIRE(row_lo >= 0 && row_hi >= row_lo && cols >= 1 && pitch >= cols, "bad row range / shape");
    EPI_REQUIRE(num_states >= 1 && num_states <= 127, "num_states=%d out of range", num_states);
    LineSource src;
    EPI_REQUIRE(src.open(path), "cannot open %s", path);
    std::vector<std::string> names;
    const char *p, *e;
    bool has_nl;
    int64_t row = 0;
    for (; row < row_lo; ++row) {
        const bool got = src.next_line(p, e, has_nl);
        EPI_REQUIRE(got || src.error().empty(), "%s", src.error().c_str());
        EPI_REQUIRE(got, "%s has only %lld rows, wanted rows from %lld", path, (long long)row, (long long)row_lo);
    }
    int last_id = -1;
    for (; row < row_hi; ++row) {
        const bool got = src.next_line(p, e, has_nl);
        EPI_REQUIRE(got || src.error().empty(), "%s", src.error().c_str());
        EPI_REQUIRE(got, "%s ends after %lld rows, wanted rows up to %lld", path, (long long)row, (long long)row_hi);
        const int64_t r = row - row_lo;
        int8_t* dst = out + r * pitch;
        int32_t cid = 0;
        if (int rc = parse_row(path, row, p, e, cols, num_states, dst, starts ? starts + r : nullptr,
                               ends ? ends + r : nullptr, &cid, names, last_id, chrom_id != nullptr))
            return rc;
        if (chrom_id != nullptr) chrom_id[r] = cid;
        for (int64_t jj = cols; jj < pitch; ++jj) dst[jj] = 0;
    }
    if (n_chrom_out) *n_chrom_out = (int32_t)names.size();
    return emit_names(names, chrom_names, chrom_names_cap);
}

// ---- single-pass parse of a whole file: the row count need not be known beforehand (saves the newline-count pass,
//      i.e. one of two inflate passes, which is what bounds reading a gzipped matrix) ------------------------------
namespace epi {
struct ParsedFile {
    static constexpr int64_t CHUNK_ROWS = 1 << 15;
    int32_t cols = 0;
    int64_t rows = 0;
    std::vector<std::unique_ptr<int8_t[]>> labels;      // chunks of CHUNK_ROWS x cols, not zero-filled: first touched by the parser threads
    std::vector<int64_t> starts, ends;
    std::vector<int32_t> chrom;
    std::vector<std::string> names;
};
}  // namespace epi

// Number of parser threads for one file: the inflate thread of every file being read plus its parsers should fit the
// machine, so a single file gets up to four parsers and a directory read file-parallel (session.prefetch) one per file.
static int parse_threads() {
    if (const char* e = getenv("EPI_PARSE_THREADS")) {
        const int v = atoi(e);
        if (v >= 1) return v > 16 ? 16 : v;
    }
    return std::max(1, std::min(8, (epi::cores_per_reader() + 2) / 3));
}

extern "C" int epi_tsv_parse_open(const char* path, int32_t num_states, void** handle_out, int64_t* rows_out,
                                  int32_t* cols_out, int32_t* n_chrom_out, int32_t* names_bytes_out) {
    EPI_REQUIRE(path != nullptr && handle_out != nullptr, "null pointer argument");
    EPI_REQUIRE(num_states >= 1 && num_states <= 127, "num_states=%d out of range", num_states);
    const double t_enter = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    LineSource src;
    EPI_REQUIRE(src.open(path), "cannot open %s", path);
    const double t_open = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count() - t_enter;
    std::unique_ptr<ParsedFile> pf(new ParsedFile());
    std::vector<std::pair<const char*, const char*>> lines;
    int last_id = -1;
    // The inflate thread hands over 16 MB blocks; all complete lines of a block are split here (memchr), the chromosome
    // names resolved (serial: the name table grows), and the rows -- whose indices, hence destinations, are known by now --
    // parsed by a few threads.  Parsing (4 ns per label) was the slower of the two pipelined stages; with it spread out
    // the single-stream inflate bounds the read.
    const bool dbg_t = getenv("EPI_INFLATE_DEBUG") != nullptr;
    double t_wait = 0, t_prep = 0, t_parse = 0;
    auto now_s = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double tq = now_s();
    while (src.next_batch(lines)) {
        double tb = now_s();
        t_wait += tb - tq;
        const int64_t n = (int64_t)lines.size(), r0 = pf->rows;
        if (r0 == 0) {
            int tabs = 0;
            for (const char* q = lines[0].first; q < lines[0].second; ++q) tabs += (*q == '\t');
            pf->cols = tabs + 1 - 3;
            EPI_REQUIRE(pf->cols >= 1, "%s: expected `chr start end state_1 ...` rows", path);
        }
        while ((int64_t)pf->labels.size() * ParsedFile::CHUNK_ROWS < r0 + n)
            pf->labels.emplace_back(new int8_t[(size_t)ParsedFile::CHUNK_ROWS * pf->cols]);
        pf->starts.resize((size_t)(r0 + n));
        pf->ends.resize((size_t)(r0 + n));
        pf->chrom.resize((size_t)(r0 + n));
        for (int64_t i = 0; i < n; ++i) {             // chromosome ids (the row's other fields are validated by parse_row)
            const char* p = lines[(size_t)i].first;
            const char* e = lines[(size_t)i].second;
            const char* t = static_cast<const char*>(memchr(p, '\t', (size_t)(e - p)));
            const size_t nl = t ? (size_t)(t - p) : (size_t)(e - p);
            int id = -1;
            if (last_id >= 0 && pf->names[(size_t)last_id].size() == nl && memcmp(pf->names[(size_t)last_id].data(), p, nl) == 0)
                id = last_id;
            for (size_t q = 0; id < 0 && q < pf->names.size(); ++q)
                if (pf->names[q].size() == nl && memcmp(pf->names[q].data(), p, nl) == 0) id = (int)q;
            if (id < 0) {
                if (t == nullptr) break;               // a truncated row: parse_row reports it
                id = (int)pf->names.size();
                pf->names.emplace_back(p, nl);
            }
            pf->chrom[(size_t)(r0 + i)] = last_id = id;
        }
        double tc = now_s();
        t_prep += tc - tb;
        const int nt = (int)std::min<int64_t>(parse_threads(), std::max<int64_t>(1, n / 256));
        std::vector<std::string> errs((size_t)nt);
        std::vector<int64_t> err_row((size_t)nt, -1);
        auto work = [&](int t) {
            std::vector<std::string> no_names;
            int no_last = -1;
            int32_t cid = 0;
            for (int64_t i = n * t / nt; i < n * (t + 1) / nt; ++i) {
                const int64_t r = r0 + i;
                int8_t* dst = pf->labels[(size_t)(r / ParsedFile::CHUNK_ROWS)].get() + (r % ParsedFile::CHUNK_ROWS) * pf->cols;
                if (parse_row(path, r, lines[(size_t)i].first, lines[(size_t)i].second, pf->cols, num_states, dst,
                              &pf->starts[(size_t)r], &pf->ends[(size_t)r], &cid, no_names, no_last, false)) {
                    errs[(size_t)t] = epi_last_error();        // the message lives in this thread's error slot
                    err_row[(size_t)t] = r;
                    return;
                }
            }
        };
        if (nt == 1) {
            work(0);
        } else {
            std::vector<std::thread> pool;
            for (int t = 0; t < nt; ++t) pool.emplace_back(work, t);
            for (auto& th : pool) th.join();
        }
        for (int t = 0; t < nt; ++t)                  // threads own ascending row ranges: the first failure is the lowest row
            if (err_row[(size_t)t] >= 0) {
                set_error("%s", errs[(size_t)t].c_str());
                return 2;
            }
        pf->rows = r0 + n;
        tq = now_s();
        t_parse += tq - tc;
    }
    if (dbg_t)
        fprintf(stderr, "[epi reader] open (load, chunk starts, first text) %.3f s; parse loop: waiting for text %.3f s, line split + ids %.3f s, "
                "row parse %.3f s\n", t_open, t_wait, t_prep, t_parse);
    EPI_REQUIRE(src.error().empty(), "%s", src.error().c_str());
    size_t nb = 0;
    for (const std::string& s : pf->names) nb += s.size() + 1;
    if (rows_out) *rows_out = pf->rows;
    if (cols_out) *cols_out = pf->cols;
    if (n_chrom_out) *n_chrom_out = (int32_t)pf->names.size();
    if (names_bytes_out) *names_bytes_out = (int32_t)nb;
    *handle_out = pf.release();
    return 0;
}

extern "C" int epi_tsv_parse_fetch(void* handle, int64_t row_lo, int64_t row_hi, int8_t* out, int64_t pitch, int64_t* starts,
                                   int64_t* ends, int32_t* chrom_id, char* chrom_names, int32_t chrom_names_cap) {
    ParsedFile* pf = static_cast<ParsedFile*>(handle);
    EPI_REQUIRE(pf != nullptr, "null handle");
    EPI_REQUIRE(row_lo >= 0 && row_hi >= row_lo && row_hi <= pf->rows, "row range [%lld, %lld) outside the %lld parsed rows",
                (long long)row_lo, (long long)row_hi, (long long)pf->rows);
    EPI_REQUIRE(row_hi == row_lo || (out != nullptr && pitch >= pf->cols), "bad output buffer");
    auto copy_rows = [&](int64_t lo, int64_t hi) {
        for (int64_t r = lo; r < hi; ++r) {
            const int8_t* src = pf->labels[(size_t)(r / ParsedFile::CHUNK_ROWS)].get() + (r % ParsedFile::CHUNK_ROWS) * pf->cols;
            int8_t* dst = out + (r - row_lo) * pitch;
            memcpy(dst, src, (size_t)pf->cols);
            if (pitch > pf->cols) memset(dst + pf->cols, 0, (size_t)(pitch - pf->cols));
        }
    };
    // large matrices: the copy into the caller's (possibly freshly allocated, not yet touched) buffer on a few threads
    const int64_t nrows = row_hi - row_lo;
    const int nt = nrows * pitch >= (32ll << 20) ? parse_threads() : 1;
    if (nt <= 1) {
        copy_rows(row_lo, row_hi);
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < nt; ++t) pool.emplace_back(copy_rows, row_lo + nrows * t / nt, row_lo + nrows * (t + 1) / nt);
        for (auto& th : pool) th.join();
    }
    const size_t n = (size_t)(row_hi - row_lo);
    if (starts && n) memcpy(starts, pf->starts.data() + row_lo, n * sizeof(int64_t));
    if (ends && n) memcpy(ends, pf->ends.data() + row_lo, n * sizeof(int64_t));
    if (chrom_id && n) memcpy(chrom_id, pf->chrom.data() + row_lo, n * sizeof(int32_t));
    return emit_names(pf->names, chrom_names, chrom_names_cap);
}

extern "C" int epi_tsv_parse_close(void* handle) {
    delete static_cast<ParsedFile*>(handle);
    return 0;
}

// ---- score text (`chr \t start \t end \t K decimal fields`, the files epi_write_scores_gz / scores.writeScores produce)
//      back into float64: replaces the pandas read of similaritySearch_max_mean.readScores (:51-74) ---------------------
namespace epi {
struct ScoreFile {
    static constexpr int64_t CHUNK_ROWS = 1 << 15;
    int32_t cols = 0;
    int64_t rows = 0;
    std::vector<std::vector<double>> vals;        // chunks of CHUNK_ROWS x cols
    std::vector<int64_t> starts, ends;
    std::vector<int32_t> chrom;
    std::vector<std::string> names;
};

// One decimal field [p, e) -> the nearest double.  Plain decimals with at most 15 significant digits are an exactly
// representable integer divided by an exactly representable power of ten, i.e. one correctly rounded division; anything
// else (exponents, nan, inf, longer mantissas) goes through strtod.
static inline bool parse_decimal(const char* p, const char* e, double* out) {
    static const double p10[] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11,
                                 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};
    const char* q = p;
    bool neg = false;
    if (q < e && (*q == '-' || *q == '+')) neg = (*q++ == '-');
    unsigned long long mant = 0;
    int digits = 0, frac = 0;
    const char* d0 = q;
    while (q < e && (unsigned)(*q - '0') <= 9 && digits < 19) {
        mant = mant * 10 + (unsigned)(*q++ - '0');
        if (mant) ++digits;
    }
    int nd = (int)(q - d0);
    if (q < e && *q == '.') {
        ++q;
        const char* f0 = q;
        while (q < e && (unsigned)(*q - '0') <= 9 && digits < 19) {
            mant = mant * 10 + (unsigned)(*q++ - '0');
            if (mant) ++digits;
        }
        frac = (int)(q - f0);
        nd += frac;
    }
    if (q == e && nd > 0 && digits <= 15 && frac <= 22) {
        const double v = (double)mant / p10[frac];
        *out = neg ? -v : v;
        return true;
    }
    char tmp[64];
    const size_t n = (size_t)(e - p);
    if (n == 0 || n >= sizeof(tmp)) return false;
    memcpy(tmp, p, n);
    tmp[n] = 0;
    char* endp = nullptr;
    *out = strtod(tmp, &endp);
    return endp == tmp + n;
}
}  // namespace epi

extern "C" int epi_scores_tsv_open(const char* path, void** handle_out, int64_t* rows_out, int32_t* cols_out,
                                   int32_t* n_chrom_out, int32_t* names_bytes_out) {
    EPI_REQUIRE(path != nullptr && handle_out != nullptr, "null pointer argument");
    LineSource src;
    EPI_REQUIRE(src.open(path), "cannot open %s", path);
    std::unique_ptr<ScoreFile> sf(new ScoreFile());
    const char *p, *e;
    bool has_nl;
    int last_id = -1;
    while (src.next_line(p, e, has_nl)) {
        if (e > p && e[-1] == '\r') --e;
        if (p == e) continue;                           // blank lines are skipped, as the pandas reader does
        const int64_t r = sf->rows;
        if (r == 0) {
            int tabs = 0;
            for (const char* q = p; q < e; ++q) tabs += (*q == '\t');
            sf->cols = tabs + 1 - 3;
            EPI_REQUIRE(sf->cols >= 1, "%s: expected `chr start end score_1 ...` rows", path);
        }
        if (r % ScoreFile::CHUNK_ROWS == 0) sf->vals.emplace_back((size_t)ScoreFile::CHUNK_ROWS * sf->cols);
        double* dst = sf->vals.back().data() + (r % ScoreFile::CHUNK_ROWS) * sf->cols;
        // chromosome
        const char* t = static_cast<const char*>(memchr(p, '\t', (size_t)(e - p)));
        EPI_REQUIRE(t != nullptr, "%s: row %lld is truncated", path, (long long)r);
        {
            const size_t nl = (size_t)(t - p);
            int id = -1;
            if (last_id >= 0 && sf->names[last_id].size() == nl && memcmp(sf->names[last_id].data(), p, nl) == 0) id = last_id;
            for (size_t i = 0; id < 0 && i < sf->names.size(); ++i)
                if (sf->names[i].size() == nl && memcmp(sf->names[i].data(), p, nl) == 0) id = (int)i;
            if (id < 0) {
                id = (int)sf->names.size();
                sf->names.emplace_back(p, nl);
            }
            sf->chrom.push_back(last_id = id);
        }
        p = t + 1;
        // start, end
        int64_t se[2] = {0, 0};
        for (int f = 0; f < 2; ++f) {
            long long v = 0;
            bool negv = false;
            if (p < e && *p == '-') {
                negv = true;
                ++p;
            }
            const char* d0 = p;
            while (p < e && *p >= '0' && *p <= '9') v = v * 10 + (*p++ - '0');
            EPI_REQUIRE(p > d0 && p < e && *p == '\t', "%s: row %lld: bad coordinate field", path, (long long)r);
            ++p;
            se[f] = negv ? -v : v;
        }
        sf->starts.push_back(se[0]);
        sf->ends.push_back(se[1]);
        // scores
        for (int j = 0; j < sf->cols; ++j) {
            EPI_REQUIRE(p <= e, "%s: row %lld has %d score columns, expected %d", path, (long long)r, j, sf->cols);
            const char* fe = static_cast<const char*>(memchr(p, '\t', (size_t)(e - p)));
            if (fe == nullptr) fe = e;
            EPI_REQUIRE(j == sf->cols - 1 || fe < e, "%s: row %lld has %d score columns, expected %d", path, (long long)r,
                        j + 1, sf->cols);
            EPI_REQUIRE(parse_decimal(p, fe, dst + j), "%s: row %lld column %d: not a number", path, (long long)r, j + 4);
            p = fe + 1;
        }
        EPI_REQUIRE(p == e + 1, "%s: row %lld has more than %d score columns", path, (long long)r, sf->cols);
        ++sf->rows;
    }
    EPI_REQUIRE(src.error().empty(), "%s", src.error().c_str());
    size_t nb = 0;
    for (const std::string& s : sf->names) nb += s.size() + 1;
    if (rows_out) *rows_out = sf->rows;
    if (cols_out) *cols_out = sf->cols;
    if (n_chrom_out) *n_chrom_out = (int32_t)sf->names.size();
    if (names_bytes_out) *names_bytes_out = (int32_t)nb;
    *handle_out = sf.release();
    return 0;
}

extern "C" int epi_scores_tsv_fetch(void* handle, double* scores, int64_t* starts, int64_t* ends, int32_t* chrom_id,
                                    char* chrom_names, int32_t chrom_names_cap) {
    ScoreFile* sf = static_cast<ScoreFile*>(handle);
    EPI_REQUIRE(sf != nullptr, "null handle");
    if (scores)
        for (int64_t r0 = 0; r0 < sf->rows; r0 += ScoreFile::CHUNK_ROWS) {
            const int64_t n = std::min<int64_t>(ScoreFile::CHUNK_ROWS, sf->rows - r0);
            memcpy(scores + r0 * sf->cols, sf->vals[(size_t)(r0 / ScoreFile::CHUNK_ROWS)].data(),
                   (size_t)n * sf->cols * sizeof(double));
        }
    const size_t n = (size_t)sf->rows;
    if (starts && n) memcpy(starts, sf->starts.data(), n * sizeof(int64_t));
    if (ends && n) memcpy(ends, sf->ends.data(), n * sizeof(int64_t));
    if (chrom_id && n) memcpy(chrom_id, sf->chrom.data(), n * sizeof(int32_t));
    return emit_names(sf->names, chrom_names, chrom_names_cap);
}

extern "C" int epi_scores_tsv_close(void* handle) {
    delete static_cast<ScoreFile*>(handle);
    return 0;
}

namespace epi {
// Rows formatted by `fmt(char* out, int64_t row) -> end` (at most row_bytes each) in blocks of 16384 rows, every block
// deflated into its own gzip member on `threads` threads, the members written in order: one valid .gz file.
template <typename Fmt>
static int write_gz_rows(const char* path, int64_t rows, size_t row_bytes, int32_t level, int32_t threads, Fmt fmt) {
    if (level < 0 || level > 9) level = 6;
    if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
    if (threads > 64) threads = 64;
    const int64_t block = 16384;
    const int64_t nblocks = (rows + block - 1) / block;
    std::vector<std::vector<unsigned char>> outs((size_t)nblocks);
    std::atomic<int64_t> next(0);
    std::atomic<int> failed(0);
    auto work = [&]() {
        std::vector<char> text;
        for (;;) {
            const int64_t bi = next.fetch_add(1);
            if (bi >= nblocks) break;
            const int64_t lo = bi * block, hi = std::min(rows, lo + block);
            text.resize((size_t)(hi - lo) * row_bytes);
            char* p = text.data();
            for (int64_t r = lo; r < hi; ++r) p = fmt(p, r);
            const size_t tlen = (size_t)(p - text.data());
            z_stream zs;
            memset(&zs, 0, sizeof(zs));
            if (deflateInit2(&zs, level, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) {     // +16: gzip member
                failed = 1;
                break;
            }
            std::vector<unsigned char>& o = outs[(size_t)bi];
            o.resize(deflateBound(&zs, (uLong)tlen) + 64);
            zs.next_in = reinterpret_cast<Bytef*>(text.data());
            zs.avail_in = (uInt)tlen;
            zs.next_out = o.data();
            zs.avail_out = (uInt)o.size();
            const int rc = deflate(&zs, Z_FINISH);
            o.resize(zs.total_out);
            deflateEnd(&zs);
            if (rc != Z_STREAM_END) {
                failed = 1;
                break;
            }
        }
    };
    std::vector<std::thread> pool;
    const int nthreads = (int)std::min<int64_t>(threads, std::max<int64_t>(nblocks, 1));
    for (int t = 0; t < nthreads; ++t) pool.emplace_back(work);
    for (auto& t : pool) t.join();
    EPI_REQUIRE(!failed, "zlib deflate failed while writing %s", path);
    FILE* f = fopen(path, "wb");
    EPI_REQUIRE(f != nullptr, "cannot open %s for writing", path);
    bool ok = true;
    if (nblocks == 0) {
        // an empty gzip member so that the file is a valid .gz holding no text
        static const unsigned char empty_gz[20] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 3, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        ok = fwrite(empty_gz, 1, sizeof(empty_gz), f) == sizeof(empty_gz);
    }
    for (auto& o : outs) ok = ok && (fwrite(o.data(), 1, o.size(), f) == o.size());
    ok = (fclose(f) == 0) && ok;
    EPI_REQUIRE(ok, "short write to %s", path);
    return 0;
}

// Pointers to `count` consecutive NUL-terminated strings.
static std::vector<const char*> split_names(const char* p, int count) {
    std::vector<const char*> names;
    for (int i = 0; i < count; ++i) {
        names.push_back(p);
        p += strlen(p) + 1;
    }
    return names;
}

static int max_chrom_id(const int32_t* chrom_id, int64_t rows) {
    int max_id = 0;
    for (int64_t r = 0; r < rows && chrom_id; ++r) max_id = std::max(max_id, (int)chrom_id[r]);
    return max_id;
}

// `chr \t start \t end` of row r
static inline char* format_location(char* p, const char* nm, int64_t start, int64_t end) {
    const size_t nl = strlen(nm);
    memcpy(p, nm, nl);
    p += nl;
    *p++ = '\t';
    p = format_i64(p, start);
    *p++ = '\t';
    return format_i64(p, end);
}
}  // namespace epi

extern "C" int epi_write_scores_gz(const char* path, const char* chrom_names, const int32_t* chrom_id,
                                   const int64_t* starts, const int64_t* ends, const float* scores, int64_t rows,
                                   int32_t K, int32_t level, int32_t threads) {
    EPI_REQUIRE(path && chrom_names && starts && ends && (scores || rows == 0), "null pointer argument");
    EPI_REQUIRE(rows >= 0 && K >= 1, "bad shape");
    const std::vector<const char*> names = split_names(chrom_names, max_chrom_id(chrom_id, rows) + 1);
    return write_gz_rows(path, rows, 64 + (size_t)K * 28, level, threads, [&](char* p, int64_t r) {
        p = format_location(p, names[chrom_id ? chrom_id[r] : 0], starts[r], ends[r]);
        const float* row = scores + r * K;
        for (int s = 0; s < K; ++s) {
            *p++ = '\t';
            p = format_5f(p, (double)row[s]);
        }
        *p++ = '\n';
        return p;
    });
}

extern "C" int epi_write_metrics_gz(const char* path, const char* chrom_names, const int32_t* chrom_id,
                                    const int64_t* starts, const int64_t* ends, const char* state_names, int32_t K,
                                    const int32_t* max_diff, const float* distance, const double* pval, const double* bh,
                                    int64_t rows, int32_t level, int32_t threads) {
    EPI_REQUIRE(path && chrom_names && starts && ends && state_names, "null pointer argument");
    EPI_REQUIRE(rows == 0 || (max_diff && distance), "null pointer argument");
    EPI_REQUIRE((pval == nullptr) == (bh == nullptr), "p-values and adjusted p-values go together");
    EPI_REQUIRE(rows >= 0 && K >= 1 && K <= EPI_MAX_STATES, "bad shape");
    for (int64_t r = 0; r < rows; ++r)
        EPI_REQUIRE(max_diff[r] >= 1 && max_diff[r] <= K, "row %lld: state %d outside 1..%d", (long long)r, max_diff[r], K);
    const std::vector<const char*> names = split_names(chrom_names, max_chrom_id(chrom_id, rows) + 1);
    const std::vector<const char*> states = split_names(state_names, K);
    size_t longest = 0;
    for (const char* s : states) longest = std::max(longest, strlen(s));
    return write_gz_rows(path, rows, 128 + longest + 64, level, threads, [&](char* p, int64_t r) {
        p = format_location(p, names[chrom_id ? chrom_id[r] : 0], starts[r], ends[r]);
        *p++ = '\t';
        const char* st = states[max_diff[r] - 1];
        const size_t sl = strlen(st);
        memcpy(p, st, sl);
        p += sl;
        *p++ = '\t';
        const float d = distance[r];
        p = format_5f(p, (double)fabsf(d));
        *p++ = '\t';
        *p++ = d >= 0.f ? '+' : '-';
        if (pval) p += sprintf(p, "\t%.5e\t%.5e", pval[r], bh[r]);
        *p++ = '\n';
        return p;
    });
}

// ---- ChromHMM `-printstatebyline` files -> matrix: the native form of bin/preprocess_data_ChromHMM.sh (SURVEY.md 8f, row f3).
//      One file per biosample and chromosome: line 1 `<biosample> <chr>`, line 2 `MaxState E`, then one state label per 200 bp
//      bin.  The script pastes the files of a chromosome side by side and prefixes every row with `chr, start, end`
//      (preprocess_data_ChromHMM.sh:34-49).  epi_statebyline_read parses ONE file straight into a column of the int8 matrix
//      (no text matrix in between); epi_write_matrix_tsv writes the script's text for callers that want the file. ----------
extern "C" int epi_statebyline_read(const char* path, int8_t* out, int64_t stride, int64_t cap_rows, int32_t num_states,
                                    int64_t* rows_out, char* chrom_out, int32_t chrom_cap) {
    EPI_REQUIRE(path != nullptr && rows_out != nullptr, "null pointer argument");
    EPI_REQUIRE(out == nullptr || stride >= 1, "bad stride");
    EPI_REQUIRE(num_states >= 1 && num_states <= 127, "num_states=%d out of range", num_states);
    LineSource src;
    EPI_REQUIRE(src.open(path), "cannot open %s", path);
    const char *p, *e;
    bool has_nl;
    int64_t line = 0, rows = 0;
    while (src.next_line(p, e, has_nl)) {
        if (e > p && e[-1] == '\r') --e;
        ++line;
        if (line == 1) {
            // `<biosample> <chr>`: the chromosome is the second whitespace-separated field (awk's $2 of the pasted line)
            const char* q = p;
            while (q < e && *q != '\t' && *q != ' ') ++q;
            while (q < e && (*q == '\t' || *q == ' ')) ++q;
            const char* c0 = q;
            while (q < e && *q != '\t' && *q != ' ') ++q;
            EPI_REQUIRE(q > c0, "%s: the first line does not name a chromosome (`<biosample> <chr>` expected)", path);
            if (chrom_out != nullptr) {
                EPI_REQUIRE((int64_t)(q - c0) + 1 <= (int64_t)chrom_cap, "chromosome name buffer too small");
                memcpy(chrom_out, c0, (size_t)(q - c0));
                chrom_out[q - c0] = 0;
            }
            continue;
        }
        if (line == 2) continue;                                   // `MaxState E`
        if (p == e && !has_nl) break;
        unsigned v = 0;
        const char* q = p;
        EPI_REQUIRE(q < e, "%s: line %lld is empty (a state label expected)", path, (long long)line);
        while (q < e && (unsigned)(*q - '0') <= 9 && v <= 1000) v = v * 10 + (unsigned)(*q++ - '0');
        EPI_REQUIRE(q == e, "%s: line %lld: state label is not an integer", path, (long long)line);
        EPI_REQUIRE(v >= 1 && v <= (unsigned)num_states, "%s: line %lld: state %u outside 1..%d", path, (long long)line, v, num_states);
        if (out != nullptr) {
            EPI_REQUIRE(rows < cap_rows, "%s has more than %lld bins", path, (long long)cap_rows);
            out[rows * stride] = (int8_t)(v - 1);
        }
        ++rows;
    }
    EPI_REQUIRE(src.error().empty(), "%s", src.error().c_str());
    EPI_REQUIRE(line >= 2, "%s: two header lines expected", path);
    *rows_out = rows;
    return 0;
}

// `chrom \t start \t end \t label_1 .. label_C` per bin, start = (first_bin + r) * bin_size, labels 1-based: the text of the
// reference's input matrices (README.md:286-292).  gz_level < 0: plain text; else gzip members of 4096 rows at that level.
extern "C" int epi_write_matrix_tsv(const char* path, const char* chrom, const int8_t* m, int64_t rows, int32_t cols,
                                    int64_t pitch, int64_t bin_size, int64_t first_bin, int32_t gz_level, int32_t threads) {
    EPI_REQUIRE(path && chrom && (m || rows == 0), "null pointer argument");
    EPI_REQUIRE(rows >= 0 && cols >= 1 && pitch >= cols && bin_size >= 1, "bad shape");
    if (gz_level > 9) gz_level = 9;
    if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
    if (threads > 64) threads = 64;
    const int64_t block = 4096;
    const int64_t nblocks = (rows + block - 1) / block;
    const size_t clen = strlen(chrom);
    FILE* f = fopen(path, "wb");
    EPI_REQUIRE(f != nullptr, "cannot open %s for writing", path);
    // blocks are produced by a pool in waves of `threads * 4` and written in order, so that memory stays bounded
    std::atomic<int> failed(0);
    bool ok = true;
    const int64_t wave = (int64_t)threads * 4;
    std::vector<std::vector<unsigned char>> outs((size_t)wave);
    for (int64_t w0 = 0; w0 < nblocks && ok && !failed; w0 += wave) {
        const int64_t w1 = std::min(nblocks, w0 + wave);
        std::atomic<int64_t> next(w0);
        auto work = [&]() {
            std::vector<char> text;
            for (;;) {
                const int64_t bi = next.fetch_add(1);
                if (bi >= w1) break;
                const int64_t lo = bi * block, hi = std::min(rows, lo + block);
                text.resize((size_t)(hi - lo) * (clen + 48 + (size_t)cols * 4));
                char* p = text.data();
                for (int64_t r = lo; r < hi; ++r) {
                    memcpy(p, chrom, clen);
                    p += clen;
                    *p++ = '\t';
                    p = format_i64(p, (first_bin + r) * bin_size);
                    *p++ = '\t';
                    p = format_i64(p, (first_bin + r + 1) * bin_size);
                    const int8_t* row = m + r * pitch;
                    for (int32_t c = 0; c < cols; ++c) {
                        const unsigned v = (unsigned)(row[c] + 1);          // 1 .. 128
                        *p++ = '\t';
                        if (v >= 100) *p++ = (char)('0' + v / 100);
                        if (v >= 10) *p++ = (char)('0' + (v / 10) % 10);
                        *p++ = (char)('0' + v % 10);
                    }
                    *p++ = '\n';
                }
                const size_t tlen = (size_t)(p - text.data());
                std::vector<unsigned char>& o = outs[(size_t)(bi - w0)];
                if (gz_level < 0) {
                    o.assign(text.data(), text.data() + tlen);
                    continue;
                }
                z_stream zs;
                memset(&zs, 0, sizeof(zs));
                if (deflateInit2(&zs, gz_level, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) {
                    failed = 1;
                    break;
                }
                o.resize(deflateBound(&zs, (uLong)tlen) + 64);
                zs.next_in = reinterpret_cast<Bytef*>(text.data());
                zs.avail_in = (uInt)tlen;
                zs.next_out = o.data();
                zs.avail_out = (uInt)o.size();
                const int rc = deflate(&zs, Z_FINISH);
                o.resize(zs.total_out);
                deflateEnd(&zs);
                if (rc != Z_STREAM_END) {
                    failed = 1;
                    break;
                }
            }
        };
        std::vector<std::thread> pool;
        const int nt = (int)std::min<int64_t>(threads, w1 - w0);
        for (int t = 0; t < nt; ++t) pool.emplace_back(work);
        for (auto& t : pool) t.join();
        for (int64_t bi = w0; bi < w1 && !failed; ++bi) {
            std::vector<unsigned char>& o = outs[(size_t)(bi - w0)];
            ok = ok && (fwrite(o.data(), 1, o.size(), f) == o.size());
        }
    }
    if (nblocks == 0 && gz_level >= 0) {
        static const unsigned char empty_gz[20] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 3, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        ok = fwrite(empty_gz, 1, sizeof(empty_gz), f) == sizeof(empty_gz);
    }
    ok = (fclose(f) == 0) && ok;
    EPI_REQUIRE(!failed, "zlib deflate failed while writing %s", path);
    EPI_REQUIRE(ok, "short write to %s", path);
    return 0;
}

// columns src[c][0..rows) (contiguous, src_stride bytes apart) -> dst[r * pitch + c], c < cols: a group of columns of a pitched
// matrix (dst may point at any column of it; bytes of a row outside [0, cols) are not touched).
// Blocked so that both sides are touched a cache line at a time; row blocks over a few threads.
extern "C" int epi_columns_to_rows(const int8_t* src, int64_t src_stride, int32_t cols, int64_t rows, int8_t* dst, int64_t pitch,
                                   int32_t threads) {
    EPI_REQUIRE((src && dst) || rows == 0 || cols == 0, "null pointer argument");
    EPI_REQUIRE(cols >= 0 && rows >= 0 && pitch >= cols && src_stride >= rows, "bad shape");
    if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
    if (threads > 64) threads = 64;
    constexpr int64_t RB = 256, CB = 64;
    const int64_t nblocks = (rows + RB - 1) / RB;
    std::atomic<int64_t> next(0);
    auto work = [&]() {
        for (;;) {
            const int64_t b = next.fetch_add(1);
            if (b >= nblocks) break;
            const int64_t r0 = b * RB, r1 = std::min(rows, r0 + RB);
            for (int64_t c0 = 0; c0 < cols; c0 += CB) {
                const int64_t c1 = std::min<int64_t>(cols, c0 + CB);
                for (int64_t r = r0; r < r1; ++r) {
                    int8_t* d = dst + r * pitch;
                    for (int64_t c = c0; c < c1; ++c) d[c] = src[c * src_stride + r];
                }
            }
        }
    };
    const int nt = (int)std::min<int64_t>(threads, std::max<int64_t>(nblocks, 1));
    if (nt <= 1) {
        work();
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < nt; ++t) pool.emplace_back(work);
        for (auto& t : pool) t.join();
    }
    return 0;
}
