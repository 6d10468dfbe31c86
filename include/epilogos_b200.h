/*
 * epilogos_b200 -- C ABI of the B200 (sm_100a) implementation of the Epilogos scoring hot path.
 *
 * This header is the drop-in boundary.  The reference (meuleman/epilogos, pure Python) has no FFI; the
 * entry points below are what a binding for its hot functions would call, one per reference function
 * (file:line cited on each).  Signatures use plain pointers and sizes only -- no torch / numpy types.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; epi_last_error() returns a message for
 *     the calling thread (the Python layer raises RuntimeError with it; the reference raises Python
 *     exceptions and has no error codes, SURVEY.md section 8b).
 *   - "device pointer" = memory of the current CUDA device (cudaMalloc / torch tensor .data_ptr()).
 *     `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Device-level entry
 *     points are asynchronous on that stream; *_host entry points take host pointers, do their own
 *     H2D/D2H copies and return after the results are in the host buffers.
 *   - the state matrix is int8, 0-based (label - 1, helpers.py:154-155), bins x biosamples, row pitch in
 *     bytes.  The fast path wants pitch % 16 == 0 and a 16-byte aligned base (the packer produces that);
 *     any other pitch is repacked on the device first.  Pad bytes are never interpreted.
 *     Labels must be < num_states (the packer validates; the reference would raise IndexError).
 *   - per-bin state counts are uint16 [bins][num_states] (a count is <= biosamples <= 65535).
 *   - there is NO CPU fallback: every compute entry point fails if no sm_100 device is present.
 *   - the score entry points keep small per-device tables (constant memory, a scratch buffer); calls for one device
 *     must be stream-ordered with respect to each other (one stream, or events between streams).
 */
#ifndef EPILOGOS_B200_H
#define EPILOGOS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EPI_ABI_VERSION 1
#define EPI_MAX_STATES 32

/* ---- library / device ------------------------------------------------------------------------ */
int epi_abi_version(void);
const char* epi_last_error(void);
/* sm count, compute capability of the current device; fails when there is no CUDA device. */
int epi_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- K1: per-bin state counts ----------------------------------------------------------------
 * cnt[b][s] = #{ j < cols : x[b][j] == s }.
 * Replaces np.unique(dataArr[row], return_counts=True) in expected.py:111,152 and scores.py:341,444. */
int epi_bin_counts(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                   uint16_t* cnt_dev, void* stream);

/* ---- column groups: counts of many column subsets of one matrix (csrc/groups.cu) ----------------------------
 * A group is a list of columns of x: group g lists group_cols[group_offsets[g] .. group_offsets[g+1]) (device int32
 * arrays; offsets start at 0 and increase strictly, every column is in [0, cols); a column may appear in several groups).
 *   epi_group_counts    cnt[g][b][s] = #{ listed columns j of group g : x[b][j] == s }, uint16 [groups][bins][num_states]:
 *                       each group's block has the layout of epi_bin_counts.  The matrix is read once for all groups;
 *                       pitch and base need no alignment (an unaligned matrix is repacked first, as in epi_bin_counts).
 *   epi_gather_columns  out[b][j] = x[b][idx[j]] for j < n; bytes n .. out_pitch of a row are zero (out_pitch a
 *                       multiple of 16): the matrix of a group's columns, in the layout the kernels consume.
 * Both copy the (small) column lists to the host to validate them, which synchronises the stream. */
#define EPI_MAX_GROUPS 64
int epi_group_counts(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                     const int32_t* group_cols_dev, const int32_t* group_offsets_dev, int32_t groups, uint16_t* cnt_dev,
                     void* stream);
int epi_gather_columns(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, const int32_t* idx_dev, int32_t n,
                       int8_t* out_dev, int64_t out_pitch, void* stream);

/* ---- K2: S1 / S2 expected count tables from the per-bin counts -------------------------------
 * n1[s]    += sum_b cnt[b][s]                                   (expected.py:106-113, s1Calc)
 * n2[s][t] += sum_b cnt[b][s]*cnt[b][t] - [s==t]*cnt[b][s]      (expected.py:146-158, s2Calc)
 * Accumulates into int64 device arrays (caller zeroes them); either pointer may be NULL.
 * `width` = biosamples per row (upper bound of a count).
 * Runs as a Gram update of the count bytes on the tensor cores (tcgen05.mma kind::i8, exact int32 accumulation). */
int epi_expected_s1s2(const uint16_t* cnt_dev, int64_t bins, int32_t num_states, int32_t width,
                      int64_t* n1_dev, int64_t* n2_dev, void* stream);

/* ---- K4: normalise an int64 count table -------------------------------------------------------
 * out[i] = (float)((double)counts[i] / (double)sum(counts))     (expectedCombination.py:42) */
int epi_normalize_i64(const int64_t* counts_dev, int64_t n, float* out_dev, void* stream);

/* ---- K5: S1 / S2 scores from the per-bin counts -----------------------------------------------
 * S1: score[b][s] = o*log2(o/E1[s]), o = cnt[b][s]/width        (scores.py:339-344, 317, 550)
 * S2: score[b][t] = sum_s o_st*log2(o_st/E2[s][t]) added in order s = 0..K-1,
 *     o_st = (cnt_s*cnt_t - [s==t]cnt_s)/perms                  (scores.py:443-451, 412, 550)
 *     `width` = labels per row = the sum of a row's counts (every row has exactly this many); `perms` = C*(C-1)
 *     of the group the observation is normalised with (they differ only for the -g quirk of scores.py:397-398).
 * Terms with o == 0 or E == 0 are 0 (numpy.ma masking of klScoreND).
 * out32 (float32, the reference's stored dtype) and/or out64 (unrounded float64) may be NULL.
 * mode: EPI_SCORE_TABLE evaluates log2 through tables of log2(count) and log2(E) (default, within
 *       1e-9 relative + 1e-12 absolute of the float64 reference; for S2 the K x K mat-vec against log2 E runs on the
 *       tensor cores with log2 E in 56-bit fixed point, i.e. exactly); EPI_SCORE_DIRECT evaluates
 *       obs*log2(obs/E) term by term with a correctly rounded divide (verification path, and the path taken
 *       automatically when the expected table has zero entries). */
#define EPI_SCORE_TABLE 0
#define EPI_SCORE_DIRECT 1
int epi_scores_s1(const uint16_t* cnt_dev, int64_t bins, int32_t num_states, int32_t width,
                  const float* exp1_dev, float* out32_dev, double* out64_dev, int32_t mode, void* stream);
int epi_scores_s2(const uint16_t* cnt_dev, int64_t bins, int32_t num_states, int32_t width, int64_t perms,
                  const float* exp2_dev, float* out32_dev, double* out64_dev, int32_t mode, void* stream);
/* Diagnostic: the fixed-point image M[s][t] = round(-log2 E2[s][t] * 2^F) (uint64 [K][K], device) that the tensor-core
 * TABLE evaluation of epi_scores_s2 (width <= 2047) multiplies the counts with, and F.  M is 56-bit, F = 56 - ib where
 * -log2 E2 < 2^ib, and the kernel takes M as seven base-256 digits (kind::i8, exact int32 accumulation). */
int epi_scores_s2_fixed_point(const float* exp2_dev, int32_t num_states, int64_t perms, uint64_t* mfix_dev,
                              int32_t* fraction_bits_out, void* stream);

/* ---- K3: S3 expected counts (expected.py:165-204, s3Calc) as an int8 one-hot Gram matrix ------------
 * N3[i][j][a][c] = #{ b : x[b][i]==a and x[b][j]==c } for i != j, 0 for i == j  (int32 per worker in the
 * reference, int64 after np.sum).  Computed as G = OH^T OH with OH[b][j*K+s] = (x[b][j]==s) on the tensor
 * cores (tcgen05.mma kind::i8, int32 accumulation, upper-triangular 128x256 tiles only).
 *   epi_s3_plan      sizes: mp = padded biosamples*states, bp = padded bins, number of tiles, bytes of the
 *                    one-hot workspace (mp*bp) and of the tile workspace (tiles + tile lookup).
 *   epi_s3_onehot    x -> transposed one-hot OHT[mp][bp] (int8 0/1, 128-byte aligned).
 *   epi_s3_gram      OHT -> tile buffer (int32); accumulate != 0 adds to the buffer (bin chunks).
 *                    The tile buffer is what ranks all-reduce (integer sum) in the multi-GPU path.
 *   epi_s3_finalize  tile buffer -> counts int64 [C][C][K][K] and/or float32 frequencies
 *                    float(double(n) / double(total_bins*C*(C-1))) (expectedCombination.py:42); mirrors the
 *                    lower triangle (N3[j][i][c][a] = N3[i][j][a][c]) and zeroes the i == j blocks. */
int epi_s3_plan(int64_t bins, int32_t cols, int32_t num_states, int64_t* mp, int64_t* bp, int64_t* ntiles,
                int64_t* onehot_bytes, int64_t* tile_bytes);
int epi_s3_onehot(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                  int8_t* oht_dev, int64_t mp, int64_t bp, void* stream);
int epi_s3_gram(const int8_t* oht_dev, int64_t mp, int64_t bp, int32_t* tiles_dev, int32_t accumulate,
                void* stream);
int epi_s3_finalize(int32_t* tiles_dev, int32_t cols, int32_t num_states, int64_t mp, int64_t total_bins,
                    int64_t* counts_dev, float* exp_dev, void* stream);

/* ---- K6: S3 scores (scores.py:455-506, s3Score) ---------------------------------------------------
 * terms[i][j][a][c] = q log2(q / E3[i][j][a][c]), q = 1/(C(C-1)), 0 where E3 == 0   (scores.py:479-480)
 * score[b][s] = sum over ordered pairs i != j with x[b][j] == s of terms[i][j][x[b][i]][x[b][j]] (:496-498)
 * Both evaluated in float64 (the reference uses float32 and differs from exact arithmetic by its own
 * accumulation noise).  terms_dev is a caller-provided float64 workspace of epi_s3_terms_size() doubles filled by
 * epi_s3_terms: block (i*C + j) holds the K*K terms [a][c] of the pair, blocks are padded to an even number of
 * doubles (16-byte bulk copies) and followed by 8 zero blocks. */
int epi_s3_terms_size(int32_t cols, int32_t num_states, int64_t* doubles_out);
int epi_s3_terms(const float* exp3_dev, int32_t cols, int32_t num_states, double* terms_dev, void* stream);
int epi_scores_s3(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                  const double* terms_dev, float* out32_dev, double* out64_dev, void* stream);

/* ---- K7 / K8: paired (two-group) epilogos ------------------------------------------------------------
 * S1/S2 scores depend on a group only through its per-bin count vector, so the paired path is:
 * epi_bin_counts on A and on B; shuffled-group counts (below); epi_scores_s1/s2 on the four count arrays
 * against the expected table of the union [A | B] (helpers.py:173-179); epi_pairwise_combine.
 *   epi_shuffled_counts_perm    counts of A' = first size_a and B' = next size_b labels of the combined row
 *                               permuted by perm[b][0..cols_a+cols_b) (helpers.py:183-194; size = group widths,
 *                               or -g for both).  Bit-exact replay of a seeded reference run.
 *   epi_shuffled_counts_philox  nperm independent uniform shuffles per bin, drawn on the device from the
 *                               group counts as multivariate hypergeometric variates (float64 inversion, 53-bit
 *                               uniforms; Philox4x32-10 keyed by seed, GLOBAL bin index = bin_offset + row,
 *                               permutation: a bin's draw does not depend on how the bins are sharded);
 *                               `width` = combined biosamples (upper bound of a row's label count); outputs
 *                               are [nperm][bins][K].  The reference draws one shuffle per bin.
 *   epi_pairwise_combine        delta = score_a - score_b (float32, scores.py:223); null_dist =
 *                               sum_s d^2 * sign(sum_s d), d = null_a - null_b, float32 with numpy's pairwise
 *                               summation order (scores.py:224-232).  Either output (with its inputs) may be NULL.
 *   epi_quiescent_mask          1 where every label of both groups equals quiescent_state (scores.py:294-303);
 *                               all 0 for quiescent_state == -1. */
int epi_shuffled_counts_perm(const int8_t* xa_dev, int64_t pitch_a, int32_t cols_a, const int8_t* xb_dev,
                             int64_t pitch_b, int32_t cols_b, const int32_t* perm_dev, int64_t bins,
                             int32_t num_states, int32_t size_a, int32_t size_b, uint16_t* cnt_a_out,
                             uint16_t* cnt_b_out, void* stream);
int epi_shuffled_counts_philox(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins,
                               int32_t num_states, int32_t width, int32_t size_a, int32_t size_b, uint64_t seed,
                               int64_t bin_offset, int32_t nperm,
                               uint16_t* cnt_a_out, uint16_t* cnt_b_out, void* stream);
/* epi_shuffled_counts_philox_range  the same draws for permutations perm_offset .. perm_offset + nperm - 1 (outputs
 *                                   [nperm][bins][K]): a caller batching the permutations continues one stream.
 *                                   epi_shuffled_counts_philox is this with perm_offset 0.  perm_offset + nperm <= 2^32. */
int epi_shuffled_counts_philox_range(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins,
                                     int32_t num_states, int32_t width, int32_t size_a, int32_t size_b, uint64_t seed,
                                     int64_t bin_offset, int64_t perm_offset, int32_t nperm,
                                     uint16_t* cnt_a_out, uint16_t* cnt_b_out, void* stream);
int epi_pairwise_combine(const float* score_a, const float* score_b, const float* null_a, const float* null_b,
                         int64_t rows, int32_t num_states, float* delta_out, float* null_dist_out, void* stream);
int epi_quiescent_mask(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins, int32_t num_states,
                       int32_t cols_a, int32_t cols_b, int32_t quiescent_state, uint8_t* mask_out, void* stream);

/* ---- paired ROI stage reductions (roiAndVisualPairwise.readInData, roiAndVisualPairwise.py:339-354) ---------
 * distance[b] = sum_s d^2 * sign(sum_s d) (float32, numpy pairwise order), max_diff[b] = 1-based state with the
 * largest |d| (ties -> higher state), where d is the delta row.  With text_round_trip != 0 every delta first goes
 * through the "%.5f" text -> float64 -> float32 round trip that the reference applies by re-reading
 * pairwiseDelta_*.txt.gz (emulated arithmetically, bit-exact).  Either output may be NULL. */
int epi_pairwise_real_reduce(const float* delta_dev, int64_t rows, int32_t num_states, int32_t text_round_trip,
                             float* dist_out, int32_t* max_diff_out, void* stream);

/* ---- per-bin permutation tests of paired mode (csrc/permutations.cu) ----------------------------------------
 * For every bin b: k[b] += #{p : |null(b, p)| >= |dist[b]|}, null(b, p) = sum_s d^2 * sign(sum_s d) with
 * d = score(A'_p) - score(B'_p) (float32, numpy pairwise order: what epi_pairwise_combine computes).  k is ADDED to, so
 * permutation blocks accumulate; no (bin, permutation) value is stored.
 *   epi_null_exceedances            from the score arrays of A' and B' of nperm shuffles, [nperm][bins][K] float32.
 *   epi_permutation_exceedances_s1  fused S1: draws permutations perm_offset .. perm_offset + nperm - 1 of every bin
 *                                   exactly as epi_shuffled_counts_philox_range, scores A' at width_a and B' at width_b
 *                                   against exp1 [K] with the values epi_scores_s1 gives in TABLE mode, and counts.
 *                                   Equal bit for bit to the composed path; width_a, width_b <= 4095. */
int epi_null_exceedances(const float* null_a_dev, const float* null_b_dev, int32_t nperm, int64_t bins,
                         int32_t num_states, const float* dist_dev, uint32_t* k_inout, void* stream);
int epi_permutation_exceedances_s1(const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins,
                                   int32_t num_states, int32_t width, int32_t size_a, int32_t size_b, uint64_t seed,
                                   int64_t bin_offset, int64_t perm_offset, int32_t nperm, const float* exp1_dev,
                                   int32_t width_a, int32_t width_b, const float* dist_dev, uint32_t* k_inout,
                                   void* stream);

/* ---- multi-group comparisons (csrc/multigroup.cu) ------------------------------------------------------------
 * G = groups (2..EPI_MAX_GROUPS) disjoint groups of biosamples; sizes: HOST array of the G group widths n_g >= 1 with
 * N = sum n_g <= 65535.  S_g [bins][K] float32 is group g's score at width n_g against the background of the union.  Per
 * bin, in float64 without fused multiply-add:
 *     m[s] = (sum_g n_g S_g[s]) / N,   T = (sum_s sum_g n_g (S_g[s] - m[s])^2) / N
 * summed over g ascending for m, and in one running sum with s outer and g inner (both ascending) for T.
 *   epi_multigroup_stat                   scores [G][bins][K] -> t_out [bins] = T, group_out = g* =
 *                                         argmax_g n_g sum_s (S_g[s] - m[s])^2, state_out = s* = argmax_s
 *                                         |S_g*[s] - m[s]| (first on ties; 0-based), sign_out = -1 if S_g*[s*] < m[s*]
 *                                         else +1.
 *   epi_multigroup_shuffled_counts_range  permutations perm_offset .. perm_offset + nperm - 1 of every bin, drawn from the
 *                                         stream of epi_shuffled_counts_philox (seed, permutation, GLOBAL bin
 *                                         bin_offset + b): for every state in order and every group in order, the
 *                                         group's count is HG(labels unassigned, labels of the state unassigned, labels
 *                                         the group still needs).  cnt [G] blocks of [bins][K], block g at
 *                                         cnt_dev + g * group_stride; out [nperm][G][bins][K].  With G = 2 and
 *                                         n_0 + n_1 the union's width, equal to epi_shuffled_counts_philox_range.
 *   epi_multigroup_null_exceedances       k[b] += #{p < nperm : T of null[p][.][b][.] >= t[b]}; null [nperm][G][bins][K]
 *                                         float32 scores of shuffled counts.
 *   epi_multigroup_exceedances_s1         fused S1: draws as epi_multigroup_shuffled_counts_range, scores group g at
 *                                         width n_g against exp1 [K] with the values epi_scores_s1 gives, and counts as
 *                                         epi_multigroup_null_exceedances.  Equal bit for bit to that composed path.
 *                                         Takes the shapes epi_multigroup_s1_fused_fits accepts.
 *   epi_multigroup_s1_fused_fits          1 if the fused S1 kernel takes this shape (every n_g <= 4095 and its tables
 *                                         fit in shared memory), else 0.  Needs no device.
 * k is ADDED to, so permutation blocks accumulate; no (bin, permutation) value is stored by the fused path. */
int epi_multigroup_stat(const float* scores_dev, int32_t groups, int64_t bins, int32_t num_states, const int32_t* sizes,
                        double* t_out, uint8_t* group_out, uint8_t* state_out, int8_t* sign_out, void* stream);
int epi_multigroup_shuffled_counts_range(const uint16_t* cnt_dev, int64_t group_stride, int32_t groups, int64_t bins,
                                         int32_t num_states, const int32_t* sizes, uint64_t seed, int64_t bin_offset,
                                         int64_t perm_offset, int32_t nperm, uint16_t* out_dev, void* stream);
int epi_multigroup_null_exceedances(const float* null_dev, int32_t groups, int32_t nperm, int64_t bins,
                                    int32_t num_states, const int32_t* sizes, const double* t_dev, uint32_t* k_inout,
                                    void* stream);
int epi_multigroup_exceedances_s1(const uint16_t* cnt_dev, int64_t group_stride, int32_t groups, int64_t bins,
                                  int32_t num_states, const int32_t* sizes, uint64_t seed, int64_t bin_offset,
                                  int64_t perm_offset, int32_t nperm, const float* exp1_dev, const double* t_dev,
                                  uint32_t* k_inout, void* stream);
int epi_multigroup_s1_fused_fits(int32_t groups, int32_t num_states, const int32_t* sizes);

/* ---- stratified permutations (csrc/strata.cu) -----------------------------------------------------------------
 * Labels are shuffled only within strata.  H = strata (1..EPI_MAX_STRATA) and G = groups (2..EPI_MAX_GROUPS); sizes: HOST
 * array [H][G] of n[h][g] >= 0, the biosamples of group g in stratum h, every stratum holding at least one, and
 * N = sum of all n[h][g] <= 65535.  cnt [H] blocks of [bins][K] uint16, block h at cnt_dev + h * stratum_stride (>= bins *
 * K): stratum h's counts over the row being shuffled.  The draw of (bin b, permutation p) takes the stream of
 * epi_shuffled_counts_philox (seed, p, GLOBAL bin bin_offset + b) and runs, for h = 0 .. H-1 in order on that stream, the
 * draw of epi_multigroup_shuffled_counts_range on stratum h's counts with sizes n[h][.]; group g's count is the sum over
 * the strata.  With H = 1 both entry points equal their unstratified counterparts bit for bit.  perm_offset + nperm <=
 * 2^32.  The sizes reach the device by one cudaMemcpyAsync (from the caller's pageable array) or in the kernel's
 * parameters.
 *   epi_stratified_shuffled_counts_range  out [nperm][G][bins][K] uint16.  Return code 2 when the largest stratum's
 *                                         sampler tables exceed shared memory (about 12,600 biosamples in one stratum
 *                                         at G = 2).
 *   epi_stratified_exceedances_s1         fused paired S1 (G = 2, sizes [H][2]): per (bin, permutation) A' = the group-0
 *                                         counts of the draw summed over the strata, B' = cnt_a + cnt_b - A', scored at
 *                                         width_a / width_b (covering sum_h n[h][0] / sum_h n[h][1], at most 4095) against
 *                                         exp1 [K] with the values epi_scores_s1 gives in TABLE mode;
 *                                         k[b] += #{p : |null(b, p)| >= |dist[b]|}, as epi_permutation_exceedances_s1.
 *                                         cnt_a + cnt_b must equal the sum of the strata's counts.  Equal bit for bit to
 *                                         the composed path (epi_stratified_shuffled_counts_range, epi_scores_s1,
 *                                         epi_null_exceedances). */
#define EPI_MAX_STRATA 64
int epi_stratified_shuffled_counts_range(const uint16_t* cnt_dev, int64_t stratum_stride, int32_t strata, int64_t bins,
                                         int32_t num_states, const int32_t* sizes, int32_t groups, uint64_t seed,
                                         int64_t bin_offset, int64_t perm_offset, int32_t nperm, uint16_t* out_dev,
                                         void* stream);
int epi_stratified_exceedances_s1(const uint16_t* cnt_dev, int64_t stratum_stride, int32_t strata, const int32_t* sizes,
                                  const uint16_t* cnt_a_dev, const uint16_t* cnt_b_dev, int64_t bins, int32_t num_states,
                                  uint64_t seed, int64_t bin_offset, int64_t perm_offset, int32_t nperm,
                                  const float* exp1_dev, int32_t width_a, int32_t width_b, const float* dist_dev,
                                  uint32_t* k_inout, void* stream);

/* ---- whole-genome label permutations: the region null (csrc/label_permutations.cu) -----------------------------
 *   epi_split_counts  counts of the groups of nsplit column splits of one matrix x (cols <= 65535, any pitch and
 *                     alignment).  members_dev (device) holds nsplit x (groups - 1) column bitsets of ceil(cols / 64)
 *                     uint64 words (column j is bit j % 64 of word j / 64); group groups - 1 of a split is the complement
 *                     of the others.  cnt[p][g][b][s] = #{ columns j of group g of split p : x[b][j] == s }, uint16: block
 *                     (p, g) starts at cnt_dev + (p * groups + g) * stride, stride = bins * num_states rounded up to a
 *                     multiple of 8, and has the layout of epi_bin_counts, 16-byte aligned (cnt_dev must be).  groups in
 *                     [2, EPI_MAX_GROUPS].  The bitsets are copied to the host and validated (which synchronises the
 *                     stream): a bit at or above cols, or a column in two groups of a split, is rejected.
 *   epi_window_max    for each row p < nrows of stat (dtype 0: float32, 1: float64; row p at stat_dev + p * row_stride
 *                     elements, n values): max_inout[p] = max(max_inout[p], max_{0 <= i <= n - W} sum_{j < W}
 *                     q(stat[p][i + j])) with q(x) = rint(x * 2^24) (round half to even) as int64 and W = window in
 *                     [1, 16384].  Rows with n < W are left unchanged.  Every value must be finite with 0 <= x < 2^24
 *                     (-0.0 included); otherwise return code 2 and a message naming one offending (row, index).
 *                     Synchronises the stream. */
int epi_split_counts(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                     const uint64_t* members_dev, int32_t nsplit, int32_t groups, uint16_t* cnt_dev, void* stream);
int epi_window_max(const void* stat_dev, int32_t dtype, int64_t nrows, int64_t row_stride, int64_t n, int32_t window,
                   int64_t* max_inout_dev, void* stream);

/* ---- paired statistics stage (roiAndVisualPairwise.py:177-242, csrc/pairwise_stats.cu) -----------------------
 *   epi_null_compact       the null distances of the bins whose quiescent flag is 0 (all bins when quiescent_dev is NULL),
 *                          stable order, every permutation: null_dev float32 [nperm][bins] -> pool_out [nperm][count]
 *                          (sized nperm * bins by the caller), *count_out_dev (device int64) = count.  workspace_dev holds
 *                          epi_null_compact_workspace_size(bins) bytes.
 *   epi_null_subsample     trial t < trials takes the first `size` images of a keyed pseudo-random permutation of [0, n)
 *                          (cycle-walking Feistel network, Philox4x32-10 rounds keyed by (seed, t)): size distinct indices
 *                          per trial.  idx_out int32 [trials][size] and/or samples_out float32 [trials][size] = pool[idx].
 *   epi_gennorm_fit        per trial, scipy.stats.gennorm.fit (rv_continuous.fit) of the `size` samples of that trial:
 *                          optimize.fmin (Nelder-Mead, xatol = fatol = 1e-4, 600 iterations / evaluations) on
 *                          _penalized_nnlf over (beta, loc, scale) from _fitstart (1, mean, std / sqrt(2)).  params_out
 *                          float64 [trials][4] = beta, loc, scale, NLL of the best vertex (returned even when not converged);
 *                          status_out int32 [trials][2] = iterations, converged (0/1).  Bit-reproducible run to run.
 *   epi_gennorm_pvalues    p[i] = Q(1/beta, (|x[i] - loc| / scale)^beta), the regularized upper incomplete gamma in float64
 *                          (= the two-sided 2 min(cdf, sf) of gennorm without the 1 - cdf cancellation); 1 at x == loc.
 *   epi_bh_adjust          Benjamini-Hochberg (statsmodels multipletests fdr_bh): p sorted ascending (p >= 0), p_sorted /
 *                          (rank / n), reverse cumulative minimum, clipped at 1, in input order.  workspace_dev holds
 *                          epi_bh_workspace_size(n) bytes; n < 2^31. */
int epi_null_compact_workspace_size(int64_t bins, int64_t* bytes_out);
int epi_null_compact(const float* null_dev, const uint8_t* quiescent_dev, int64_t bins, int32_t nperm, float* pool_out,
                     int64_t* count_out_dev, void* workspace_dev, int64_t workspace_bytes, void* stream);
int epi_null_subsample(const float* pool_dev, int64_t n, int32_t trials, int32_t size, uint64_t seed, int32_t* idx_out,
                       float* samples_out, void* stream);
int epi_gennorm_fit(const float* samples_dev, int32_t trials, int32_t size, double* params_out, int32_t* status_out,
                    void* stream);
int epi_gennorm_pvalues(const float* x_dev, int64_t n, double beta, double loc, double scale, double* p_out,
                        void* stream);
int epi_bh_workspace_size(int64_t n, int64_t* bytes_out);
int epi_bh_adjust(const double* p_dev, int64_t n, double* q_out, void* workspace_dev, int64_t workspace_bytes,
                  void* stream);

/* ---- whole path with HOST buffers (what expected.main -> expectedCombination.main -> scores.main
 *      compute for one in-memory matrix; run.py:196,231,246) ------------------------------------
 * x_host: int8 [bins][pitch] (any pitch >= cols; pinned memory makes the copies asynchronous).
 * saliency 1 or 2.  counts_host: int64 [K] or [K*K] (the temp_exp_freq payload), exp_host: float32
 * same shape (the exp_freq payload), scores_host: float32 [bins][K].  Any output may be NULL.
 * H2D of the matrix is chunked and overlapped with the count kernel. */
int epi_single_host(const int8_t* x_host, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states,
                    int32_t saliency, int64_t* counts_host, float* exp_host, float* scores_host);

/* ---- bit-packed transport layout of the state matrix (csrc/packbits.cu) ----------------------------
 * The kernels compute on the int8 matrix, but a label carries 5 bits (4 for <= 16 states) and epi_single_host is bound by
 * the PCIe copy of the matrix.  The packed layout is what the reader side can hand over instead: a row is
 * ceil(cols / 8) groups of 8 labels in `bits` bytes (label j in bits [bits*j, bits*(j+1)) of the little-endian group),
 * rows packed_pitch bytes apart (epi_packed_pitch: a multiple of 16).
 *   epi_packed_bits / epi_packed_pitch   bits for a state model, row pitch for a width
 *   epi_pack_states_host                 int8 host matrix -> packed host matrix (CPU threads; threads <= 0: all cores)
 *   epi_pack_states / epi_unpack_states  the same conversion on the device, both directions
 *   epi_single_host_packed               epi_single_host with the matrix in the packed layout: packed chunks cross PCIe and
 *                                        are expanded on the device right before the count kernel (helpers.py:150-160 hands
 *                                        the reference an int64 array; this is the narrowest exact form of the same labels) */
int epi_packed_bits(int32_t num_states);
int64_t epi_packed_pitch(int32_t cols, int32_t bits);
int epi_pack_states_host(const int8_t* x_host, int64_t bins, int32_t cols, int64_t pitch, int32_t bits,
                         uint8_t* packed_host, int64_t packed_pitch, int32_t threads);
int epi_pack_states(const int8_t* x_dev, int64_t bins, int32_t cols, int64_t pitch, int32_t bits, uint8_t* packed_dev,
                    int64_t packed_pitch, void* stream);
int epi_unpack_states(const uint8_t* packed_dev, int64_t bins, int32_t cols, int32_t bits, int64_t packed_pitch,
                      int8_t* x_dev, int64_t pitch, void* stream);
int epi_single_host_packed(const uint8_t* packed_host, int64_t bins, int32_t cols, int64_t packed_pitch, int32_t bits,
                           int32_t num_states, int32_t saliency, int64_t* counts_host, float* exp_host, float* scores_host);

/* ---- S3 and paired mode with HOST buffers ----------------------------------------------------------
 * epi_s3_host      expected.main (S3) -> expectedCombination.main -> scores.main (S3) for one in-memory matrix
 *                  (expected.py:165-204, expectedCombination.py:42, scores.py:455-506): exp_host float32 [C][C][K][K] or
 *                  NULL, scores_host float32 [bins][K] or NULL.
 * epi_paired_host  calculateScoresPairwise for one pair of in-memory matrices (scores.py:172-256): expected table of the
 *                  union [A | B] (helpers.py:173-179), delta = score(A) - score(B), quiescence mask, and nperm
 *                  device-drawn null shuffles per bin (the reference draws one) with their signed squared distances.
 *                  group_size -1 = the groups' own widths, else -g (clipped like the reference's slices, helpers.py:190-194);
 *                  bin_offset = global index of row 0 (keys the random streams).  Outputs (any may be NULL): counts int64 /
 *                  exp float32 [K] or [K][K], delta float32 [bins][K], null float32 [nperm][bins], quiescent uint8 [bins].
 *                  Null row p of a bin is permutation p of the stream keyed by (seed, bin_offset + row), the draw
 *                  epi_shuffled_counts_philox_range makes, whatever batches the call splits the permutations into. */
int epi_s3_host(const int8_t* x_host, int64_t bins, int32_t cols, int64_t pitch, int32_t num_states, float* exp_host,
                float* scores_host);
int epi_paired_host(const int8_t* xa_host, int64_t pitch_a, int32_t cols_a, const int8_t* xb_host, int64_t pitch_b,
                    int32_t cols_b, int64_t bins, int32_t num_states, int32_t saliency, int32_t quiescent_state,
                    int32_t group_size, uint64_t seed, int64_t bin_offset, int32_t nperm, int64_t* counts_host,
                    float* exp_host, float* delta_host, float* null_host, uint8_t* quiescent_host);

/* ---- host-side I/O either side of the kernels (no GPU needed) -------------------------------------
 * epi_tsv_shape       rows = number of newline characters (helpers.countRows, helpers.py:80-99), cols = biosample
 *                     columns of the first line (fields - 3).  Plain or gzip files.
 * epi_pack_tsv        rows [row_lo, row_hi) of `chr start end s_1 .. s_C` (README.md:286-292) -> int8 labels-1 into
 *                     out[row][pitch] (pad bytes zeroed), start/end per row, chromosome ids per row plus the distinct
 *                     names as consecutive NUL-terminated strings.  Replaces the pandas parse of helpers.readStates
 *                     (helpers.py:150-168) and of scores.py:161.  Labels outside 1..num_states are an error.
 * epi_write_scores_gz `chr\tstart\tend\t` + K x "%.5f" per row through gzip (scores.writeScores, scores.py:509-536);
 *                     decompressed text is byte-identical to the reference's.  level 0-9 (else 6), threads <= 0 = all.
 * epi_tsv_parse_*     the same parse in ONE pass over the file when the row count is not known beforehand (inflating a
 *                     gzipped matrix is what bounds reading it): _open parses the whole file into a library-owned
 *                     staging area and reports rows / columns / chromosome names; _fetch copies a row range into the
 *                     caller's (pinned) buffers exactly as epi_pack_tsv would have written them; _close frees it. */
/* Diagnostic: the decompressed byte stream the parsers see for `path` (gzip through the library's own DEFLATE decoder,
 * csrc/fast_inflate.h, with CRC-32 / ISIZE checks per member -- large files on several threads at once,
 * csrc/parallel_inflate.h; zlib with EPI_ZLIB_INFLATE=1; plain files as they are).
 * Copies at most cap bytes to out (NULL allowed); *n_out = total length. */
int epi_inflate_file(const char* path, uint8_t* out, int64_t cap, int64_t* n_out);
/* Diagnostic: how the calling thread's last finished read was inflated.  out4[0] = 0 zlib / plain file, 1 the sequential
 * native decoder, 2 the parallel decoder, 3 the parallel decoder gave up midway (zlib finished the file);
 * out4[1..3] = chunks of the compressed file, chunks in which a block / member start was found, chunks accepted. */
int epi_reader_stats(int64_t* out4);
/* Hint: the caller is about to read `files` inputs concurrently (session.prefetch) while `ranks` processes of this host
 * read at the same time (0: all LOCAL_WORLD_SIZE of them; 1 when one rank reads for everybody): every reader then takes
 * its share of the cores for its inflate and parser threads from the start.  (0, 0) clears the hint. */
int epi_reader_concurrency(int32_t files, int32_t ranks);
/* Diagnostic: the threads a reader opened now would use for its gzip stream (1 = sequential decoder) and for row parsing. */
int epi_reader_threads(int32_t* inflate_out, int32_t* parse_out);
int epi_tsv_shape(const char* path, int64_t* rows_out, int32_t* cols_out);
int epi_tsv_parse_open(const char* path, int32_t num_states, void** handle_out, int64_t* rows_out, int32_t* cols_out,
                       int32_t* n_chrom_out, int32_t* names_bytes_out);
int epi_tsv_parse_fetch(void* handle, int64_t row_lo, int64_t row_hi, int8_t* out, int64_t pitch, int64_t* starts,
                        int64_t* ends, int32_t* chrom_id, char* chrom_names, int32_t chrom_names_cap);
int epi_tsv_parse_close(void* handle);
int epi_pack_tsv(const char* path, int64_t row_lo, int64_t row_hi, int32_t cols, int32_t num_states, int8_t* out,
                 int64_t pitch, int64_t* starts, int64_t* ends, int32_t* chrom_id, char* chrom_names,
                 int32_t chrom_names_cap, int32_t* n_chrom_out);
/* Score text (`chr start end score_1 .. score_K`, what epi_write_scores_gz / scores.writeScores produce) back into
 * float64 rows: replaces the pandas read of similaritySearch_max_mean.readScores (similaritySearch_max_mean.py:51-74).
 * One pass: open parses the whole file (rows, columns, chromosome-name bytes out), fetch copies scores [rows][cols],
 * starts, ends, chromosome ids and the NUL-separated name table, close frees the handle.  Decimal fields convert to
 * the nearest double. */
int epi_scores_tsv_open(const char* path, void** handle_out, int64_t* rows_out, int32_t* cols_out, int32_t* n_chrom_out,
                        int32_t* names_bytes_out);
int epi_scores_tsv_fetch(void* handle, double* scores, int64_t* starts, int64_t* ends, int32_t* chrom_id,
                         char* chrom_names, int32_t chrom_names_cap);
int epi_scores_tsv_close(void* handle);
int epi_write_scores_gz(const char* path, const char* chrom_names, const int32_t* chrom_id, const int64_t* starts,
                        const int64_t* ends, const float* scores, int64_t rows, int32_t num_states, int32_t level,
                        int32_t threads);
/* pairwiseMetrics text through gzip, one line per bin: `chr \t start \t end \t <state name of max_diff (1-based)> \t
 * "%.5f" of |distance| \t + or - (sign of distance) [\t "%.5e" p \t "%.5e" bh]`; the last two columns only when pval and
 * bh are both given.  state_names: NUL-separated names of states 1..K.  Same deflate path as epi_write_scores_gz. */
int epi_write_metrics_gz(const char* path, const char* chrom_names, const int32_t* chrom_id, const int64_t* starts,
                         const int64_t* ends, const char* state_names, int32_t num_states, const int32_t* max_diff,
                         const float* distance, const double* pval, const double* bh, int64_t rows, int32_t level,
                         int32_t threads);
/* pairwisePermutation text through gzip, one line per bin: `chr \t start \t end \t k \t "%.5e" p \t "%.5e" bh` (k the
 * bin's exceedance count, p its permutation p-value, bh the Benjamini-Hochberg adjustment).  Same deflate path as
 * epi_write_scores_gz. */
int epi_write_permutations_gz(const char* path, const char* chrom_names, const int32_t* chrom_id, const int64_t* starts,
                              const int64_t* ends, const uint32_t* k, const double* pval, const double* bh, int64_t rows,
                              int32_t level, int32_t threads);
/* multigroupMetrics text through gzip, one line per bin: `chr \t start \t end \t "%.5e" T \t <name of group g*> \t
 * <name of state s*> \t + or - [\t k \t "%.5e" p \t "%.5e" bh]` (group and state 0-based indices into the NUL-separated
 * group_names and state_names; sign < 0 prints -); the last three columns only when k, pval and bh are all given.  Same
 * deflate path as epi_write_scores_gz. */
int epi_write_multigroup_gz(const char* path, const char* chrom_names, const int32_t* chrom_id, const int64_t* starts,
                            const int64_t* ends, const double* t, const uint8_t* group, const uint8_t* state,
                            const int8_t* sign, const char* group_names, int32_t groups, const char* state_names,
                            int32_t num_states, const uint32_t* k, const double* pval, const double* bh, int64_t rows,
                            int32_t level, int32_t threads);
/* ChromHMM `-printstatebyline` files (one per biosample and chromosome: `<biosample> <chr>`, `MaxState E`, then one label per
 * 200 bp bin) -> matrix: the native form of bin/preprocess_data_ChromHMM.sh:34-49, which pastes those files side by side.
 * epi_statebyline_read  parses ONE file into a column: out[r * stride] = label - 1 for bin r (out == NULL: count only);
 *                       *rows_out = bins in the file; chrom_out receives the chromosome named on the first line.
 * epi_write_matrix_tsv  `chrom\tstart\tend\tlabel_1..label_C` per bin (labels 1-based, start = (first_bin + r) * bin_size):
 *                       the text of the reference's input matrices (README.md:286-292); gz_level < 0 = plain text, else gzip. */
int epi_statebyline_read(const char* path, int8_t* out, int64_t stride, int64_t cap_rows, int32_t num_states, int64_t* rows_out,
                         char* chrom_out, int32_t chrom_cap);
int epi_write_matrix_tsv(const char* path, const char* chrom, const int8_t* m, int64_t rows, int32_t cols, int64_t pitch,
                         int64_t bin_size, int64_t first_bin, int32_t gz_level, int32_t threads);
/* columns src[c][0..rows) (src_stride bytes apart) -> dst[r * pitch + c], c < cols (dst may point at any column of a pitched
 * int8 matrix; other bytes of a row are not touched): the per-biosample columns of epi_statebyline_read, read contiguously,
 * into the layout the kernels consume. */
int epi_columns_to_rows(const int8_t* src, int64_t src_stride, int32_t cols, int64_t rows, int8_t* dst, int64_t pitch,
                        int32_t threads);

/* ---- region-of-interest selection over the per-bin score sums (host code) ---------------------------
 * helpers.maxMean (helpers.py:253-274) -> filter_regions maxmean (filter_regions.py:375-448): centered rolling
 * max / mean over `window` bins, windows over two chromosomes dropped, ranked by (max, mean, score) descending,
 * greedy non-overlapping pick of at most max_regions.  Outputs are in the order helpers.maxMean returns them
 * (out arrays sized max_regions): index of the window's centre row, window start / end coordinates, RollingMax,
 * RollingMean. */
int epi_roi_maxmean(const double* score, const int64_t* starts, const int64_t* ends, int64_t n, int32_t window,
                    int32_t max_regions, int64_t* out_original_idx, int64_t* out_start, int64_t* out_end,
                    double* out_rolling_max, double* out_rolling_mean, int32_t* n_out);

/* ---- similarity-search distance engine (similaritySearch_calc.runEuclideanDistance, similaritySearch_calc.py:67-123) --
 * For every ROI r (nS reduced bins x K states, row-major [R][nS][K] float64) and every window w of the reduced genome
 * ([G][K] float64):  dist[r][w] = sum_j max(0, ((-2 X[w+j].Y_r[j]) + XX[w+j]) + YY_r[j]),  w < W = G - nS + 1 -- sklearn's
 * euclidean_distances(squared=True) gathered along diagonals and summed (similaritySearch_calc.py:86-99).
 *   epi_simsearch_row_norms    XX[a] = |X[a]|^2, once per genome
 *   epi_simsearch_distances    dist for a batch of ROIs (float64 [R][W])
 *   epi_simsearch_mode_sorted  scipy.stats.mode of every row of an ASCENDING float64 [R][W] array (most frequent value,
 *                              the smallest among ties; :101): the acceptance threshold is half of it; count_dev may be NULL
 *   epi_simsearch_pick         the greedy selection (:103-123) on the device: windows in increasing distance (sorted_dev /
 *                              index_dev = sorted distances and their window indices, [R][W]), no overlap with the ROI itself
 *                              (region_start_dev, reduced bins) or an earlier pick, -1 fill after the first admissible
 *                              window farther than mode / 2; out_dev int32 [R][n_desired] */
int epi_simsearch_row_norms(const double* genome_dev, int64_t G, int32_t K, double* xx_dev, void* stream);
int epi_simsearch_distances(const double* genome_dev, const double* xx_dev, int64_t G, int32_t K, const double* rois_dev,
                            int32_t R, int32_t nS, double* dist_dev, void* stream);
int epi_simsearch_mode_sorted(const double* sorted_dev, int32_t R, int64_t W, double* mode_dev, int64_t* count_dev,
                              void* stream);
int epi_simsearch_pick(const double* sorted_dev, const int64_t* index_dev, int32_t R, int64_t W, const double* mode_dev,
                       const int64_t* region_start_dev, int32_t nS, int32_t n_desired, int32_t* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EPILOGOS_B200_H */
