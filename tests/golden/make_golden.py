"""Generate the golden fixtures in this directory by running the UNMODIFIED reference.

Run once with a checkout of the reference:   EPILOGOS_REFERENCE=/path/to/epilogos python tests/golden/make_golden.py
The reference ships no tests / golden vectors for the scoring path (SURVEY.md section 4), so the goldens
are outputs of the reference itself (expected.main -> expectedCombination.main -> scores.main through
oracle/reference_driver.py) on
  * a real-data slice: 10 biosamples x 4000 bins of chr1 built from the reference's data/ChromHMM with the
    paste recipe of bin/preprocess_data_ChromHMM.sh:34-49 (rows 100000..103999, a varied region), and
  * small seeded synthetic matrices of the benchmark shapes (C=833/K=18, C=127/K=15).
Each fixture is a compressed .npz holding the 0-based int8 input and the reference outputs.
"""
import gzip
import hashlib
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))

from oracle import reference_driver as ref            # noqa: E402
from oracle import epilogos_oracle as orc              # noqa: E402


def real_slice(lo=100000, n=4000):
    files = sorted((ref.REFERENCE_ROOT / "data" / "ChromHMM").glob("*_chr1_statebyline.txt.gz"))
    cols = []
    for f in files:
        with gzip.open(f, "rt") as g:
            lines = g.read().split("\n")
        vals = np.array([int(v) for v in lines[2:2 + lo + n] if v != ""][lo:lo + n], dtype=np.int8)
        cols.append(vals)
    return np.stack(cols, axis=1) - 1


def text_digest(text):
    return np.frombuffer(hashlib.sha256(text).digest(), dtype=np.uint8)


def single_case(name, x, k, saliencies, keep_text=True, nproc=1):
    out = {"x": x.astype(np.int8), "num_states": np.int64(k)}
    for s in saliencies:
        r = ref.run_single(x, k, s, nproc=nproc)
        out["s%d_counts" % s] = r["counts"]
        out["s%d_exp" % s] = r["exp"]
        out["s%d_scores" % s] = r["scores"]
        out["s%d_text_sha256" % s] = text_digest(r["scores_text"])
        if keep_text:
            out["s%d_text" % s] = np.frombuffer(r["scores_text"], dtype=np.uint8)
    np.savez_compressed(HERE / (name + ".npz"), **out)
    print("wrote", name, {k_: getattr(v, "shape", None) for k_, v in out.items()})


def paired_case(name, xa, xb, k, saliencies, seed, group_size=-1, quiescent_state=None):
    out = {"xa": xa.astype(np.int8), "xb": xb.astype(np.int8), "num_states": np.int64(k),
           "seed": np.int64(seed), "group_size": np.int64(group_size),
           "quiescent_state": np.int64(k - 1 if quiescent_state is None else quiescent_state)}
    for s in saliencies:
        r = ref.run_paired(xa, xb, k, s, seed, quiescent_state=quiescent_state, group_size=group_size)
        out["s%d_counts" % s] = r["counts"]
        out["s%d_exp" % s] = r["exp"]
        out["s%d_null" % s] = r["null_distances"]
        out["s%d_quiescence" % s] = r["quiescence"]
        out["s%d_delta_text" % s] = np.frombuffer(r["delta_text"], dtype=np.uint8)
    np.savez_compressed(HERE / (name + ".npz"), **out)
    print("wrote", name)


def s3_big_case(name, bins=48, cols=833, k=18, seed=11):
    """S3 at the benchmark width.  The 0.9 GB tables cannot be committed: keep sha256 digests of the
    int64 count table and float32 expected table, a strided sample of entries, and the reference scores."""
    x = orc.synth_states(bins, cols, k, seed)
    r = ref.run_single(x, k, 3)
    counts, exp = r["counts"], r["exp"]
    flat_idx = np.arange(0, counts.size, 100003, dtype=np.int64)
    out = {"x": x.astype(np.int8), "num_states": np.int64(k),
           "counts_sha256": np.frombuffer(hashlib.sha256(np.ascontiguousarray(counts).tobytes()).digest(), np.uint8),
           "exp_sha256": np.frombuffer(hashlib.sha256(np.ascontiguousarray(exp).tobytes()).digest(), np.uint8),
           "sample_idx": flat_idx, "counts_sample": counts.ravel()[flat_idx], "exp_sample": exp.ravel()[flat_idx],
           "s3_scores": r["scores"], "counts_dtype": np.array(str(counts.dtype))}
    np.savez_compressed(HERE / (name + ".npz"), **out)
    print("wrote", name)


def real_full_case():
    """BASELINE configs[0] substitute: the whole real chr1 matrix (1,246,253 bins x 10 biosamples, 18 states) assembled
    from the reference's data/ChromHMM, run through the reference's stages with 8 worker processes.  Outputs are too big to
    commit: keep the input (0.6 MB compressed), the tables, sha256 digests of the float32 score arrays and of the
    scores text, and the reference's own top-100 regions of interest (helpers.maxMean on its scores)."""
    import warnings
    x = real_slice(0, 1246253)
    out = {"x": x.astype(np.int8), "num_states": np.int64(18)}
    scores1 = None
    for s in (1, 2):
        r = ref.run_single(x, 18, s, nproc=8)
        out["s%d_counts" % s] = r["counts"]
        out["s%d_exp" % s] = r["exp"]
        out["s%d_scores_sha256" % s] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(r["scores"]).tobytes()).digest(), np.uint8)
        out["s%d_text_sha256" % s] = text_digest(r["scores_text"])
        out["s%d_scores_head" % s] = r["scores"][:2000]
        if s == 1:
            scores1 = r["scores"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from epilogos.helpers import maxMean
    n = len(scores1)
    loc = np.empty((n, 3), dtype=object)
    loc[:, 0] = "chr1"; loc[:, 1] = np.arange(n) * 200; loc[:, 2] = np.arange(n) * 200 + 200
    rois, idx = maxMean(np.concatenate((loc, scores1.sum(axis=1).reshape(n, 1)), axis=1), 50, 100)
    out.update(roi_original_idx=idx.astype(np.int64), roi_start=rois["Start"].to_numpy(np.int64),
               roi_end=rois["End"].to_numpy(np.int64), roi_rolling_max=rois["RollingMax"].to_numpy(np.float64))
    np.savez_compressed(HERE / "real10_chr1_full.npz", **out)
    print("wrote real10_chr1_full")


def roi_wide_case():
    """Region-of-interest rankings at the benchmark width (833 biosamples, 18 states) from the UNMODIFIED reference:
    expected + scores for S1 and S2 on 24,000 synthetic bins (8 worker processes), S3 on the first 160 of them, then the
    reference's own helpers.maxMean on scoreArr.sum(axis=1) (roiSingle.py:118-119) with windows of 50 bins.  The matrix is not
    stored (it is regenerated from its seed, orc.synth_states(24000, 833, 18, seed=77)); a sha256 of it guards the
    generator.  Also S2 of the 4000-bin real-data slice (10 biosamples)."""
    import warnings
    bins, cols, k, seed = 24000, 833, 18, 77
    x = orc.synth_states(bins, cols, k, seed)
    out = {"bins": np.int64(bins), "cols": np.int64(cols), "num_states": np.int64(k), "seed": np.int64(seed),
           "x_sha256": np.frombuffer(hashlib.sha256(np.ascontiguousarray(x).tobytes()).digest(), np.uint8)}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref._import_reference()
        from epilogos.helpers import maxMean

    def rank(scores, width, tag):
        n = len(scores)
        loc = np.empty((n, 3), dtype=object)
        loc[:, 0] = "chr1"; loc[:, 1] = np.arange(n) * 200; loc[:, 2] = np.arange(n) * 200 + 200
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            rois, idx = maxMean(np.concatenate((loc, scores.sum(axis=1).reshape(n, 1)), axis=1), width, 100)
        out[tag + "_roi_original_idx"] = np.asarray(idx).astype(np.int64)
        out[tag + "_roi_start"] = rois["Start"].to_numpy(np.int64)
        out[tag + "_roi_end"] = rois["End"].to_numpy(np.int64)
        out[tag + "_roi_rolling_max"] = rois["RollingMax"].to_numpy(np.float64)
        out[tag + "_scores_sha256"] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(scores).tobytes()).digest(), np.uint8)

    for s in (1, 2):
        r = ref.run_single(x, k, s, nproc=8)
        out["s%d_exp" % s] = r["exp"]
        rank(r["scores"], 50, "s%d" % s)
    r3 = ref.run_single(x[:160], k, 3, nproc=2)
    out["s3_scores"] = r3["scores"]
    rank(r3["scores"], 5, "s3")
    real = real_slice()
    r = ref.run_single(real, 18, 2)
    out["real_s2_exp"] = r["exp"]
    rank(r["scores"], 50, "real_s2")
    np.savez_compressed(HERE / "roi_wide_c833_k18.npz", **out)
    print("wrote roi_wide_c833_k18", {k_: getattr(v, "shape", None) for k_, v in out.items()})


def simsearch_case():
    """similaritySearch_calc.runEuclideanDistance of the reference (SURVEY.md 8f, row f4) on a synthetic reduced genome:
    continuous scores with a flat background on half of the bins (so that the mode of the distances exists, as it does
    for quiescent stretches of real data), ROIs = windows of the genome itself."""
    rng = np.random.default_rng(0)
    g, k, block, window = 4000, 18, 5, 25
    red = rng.random((g, k)) * rng.random((g, 1))
    red[rng.random(g) < 0.5] = 0.01
    # plant near-copies of two ROIs so that some hits pass the half-mode threshold
    starts = np.array([100, 700, 1500, 2600, 3300])
    for s, copies in ((100, (900, 2000, 3500)), (2600, (300, 1200))):
        for c in copies:
            red[c:c + window // block] = red[s:s + window // block] + rng.normal(0, 1e-3, (window // block, k))
    out = ref.run_simsearch(red, starts, window, block, 10)
    deep = ref.run_simsearch(red, starts[:2], window, block, 600)          # long lists: ends in the -1 (threshold) branch
    np.savez_compressed(HERE / "simsearch_g4000_k18.npz", reduced_genome=red, roi_starts=starts, window_bins=np.int64(window),
                        block_size=np.int64(block), n_desired=np.int64(10), indices=out, indices_deep=deep)
    print("wrote simsearch_g4000_k18", out[:, :4].tolist())
    # second shape: 15 states, windows of 3 reduced bins (blockSize 2), two chromosomes whose coordinates restart
    rng = np.random.default_rng(1)
    g, k, block, window, split = 5000, 15, 2, 6, 6000
    red = rng.random((g, k)) ** 2
    red[rng.random(g) < 0.4] = 0.005                             # flat stretches: the mode of the distances
    starts = np.array([40, 2999, 3000, 3500, 4990])              # 2999: the window straddles the chromosome boundary
    for s in starts:                                             # the ROIs themselves are not flat (no exactly tied picks:
        red[s:s + window // block] = rng.random((window // block, k)) ** 2      # their order is numpy-introsort specific)
    for s, copies in ((3500, (100, 4200)), (40, (700,))):
        for c in copies:
            red[c:c + window // block] = red[s:s + window // block] * (1 + rng.normal(0, 1e-4, (window // block, k)))
    out = ref.run_simsearch(red, starts, window, block, 25, chrom_split=split)
    np.savez_compressed(HERE / "simsearch_g5000_k15_2chrom.npz", reduced_genome=red, roi_starts=starts,
                        window_bins=np.int64(window), block_size=np.int64(block), n_desired=np.int64(25), indices=out,
                        chrom_split=np.int64(split))
    print("wrote simsearch_g5000_k15_2chrom", out[:, :4].tolist(), (out == -1).sum(axis=1).tolist())


def simsearch_prep_case():
    """similaritySearch_max_mean.main of the reference on S1 scores of REAL data (60,000 bins of chr1, 10 biosamples,
    long quiescent stretches = many exactly tied sums) and, with other window / filter settings, on a two-chromosome
    synthetic track.  The fixture keeps the scores as integers (value x 1e5: exactly what the 5-decimal text holds)."""
    import tempfile
    from oracle import simsearch_oracle as sso
    def run(name, q, chrom, starts, cfgs):
        text = "".join("%s\t%d\t%d\t%s\n" % (chrom[i], starts[i], starts[i] + 200, "\t".join("%.5f" % (v / 1e5) for v in q[i]))
                       for i in range(len(q)))
        save = dict(scores_q=q, chrom=np.array(chrom), starts=np.asarray(starts, dtype=np.int64))
        with tempfile.TemporaryDirectory() as tmp:
            path = Path(tmp) / "scores_x.txt.gz"
            with gzip.open(path, "wt", compresslevel=1) as f:
                f.write(text)
            for j, (wb, bs, wbp, fst, fsc) in enumerate(cfgs):
                r = ref.run_simsearch_prep(path, wb, bs, wbp, fst, fsc)
                assert np.array_equal(r["genome_scores"], q / 1e5)
                # the restatement against the reference, here, before the fixture is trusted
                sc = r["genome_scores"]
                sums = sso.row_sums(sc)
                assert np.array_equal(sso.reduce_genome(sc, sums, bs), r["reduced_genome"]), "reduce_genome restatement"
                save["cfg%d" % j] = np.array([wb, bs, wbp, fst], dtype=np.int64)
                save["filter_score%d" % j] = np.float64(fsc)
                save["cube_chrom%d" % j] = np.array([str(c) for c in r["cube_coords"][:, 0]])
                save["cube_start%d" % j] = r["cube_coords"][:, 1].astype(np.int64)
                save["cube_end%d" % j] = r["cube_coords"][:, 2].astype(np.int64)
                save["cube_digest%d" % j] = text_digest(np.ascontiguousarray(r["cube_scores"]).tobytes())
                save["cube_shape%d" % j] = np.array(r["cube_scores"].shape, dtype=np.int64)
                save["cube_first%d" % j] = r["cube_scores"][:3]
                save["reduced_digest%d" % j] = text_digest(np.ascontiguousarray(r["reduced_genome"]).tobytes())
                save["reduced_rows%d" % j] = np.int64(len(r["reduced_genome"]))
                print(name, "cfg", j, "regions", r["cube_scores"].shape, "reduced", r["reduced_genome"].shape)
        save["n_cfg"] = np.int64(len(cfgs))
        np.savez_compressed(HERE / (name + ".npz"), **save)
    x = real_slice(lo=100000, n=60000)
    _, sc32 = orc.expected_and_scores(x, 18, 1)
    q = np.round(sc32.astype(np.float64) * 1e5).astype(np.int32)
    run("simsearch_prep_real_chr1_60k", q, ["chr1"] * len(q), (100000 + np.arange(len(q))) * 200,
        [(125, 5, 25000, -1, -1.0), (50, 2, 10000, 0, 1.5)])
    rng = np.random.default_rng(5)
    b, k = 9003, 15                                         # not a multiple of the block size: a partial last block
    q = (np.round(rng.gamma(0.3, 1.0, (b, k)) * (rng.random((b, 1)) < 0.3), 5) * 1e5).astype(np.int32)
    chrom = ["chr1"] * 5000 + ["chrX"] * (b - 5000)
    starts = np.concatenate((np.arange(5000), np.arange(b - 5000))) * 200
    run("simsearch_prep_synth_2chrom", q, chrom, starts, [(125, 5, 25000, -1, -1.0), (25, 1, 5000, 3, 2.0), (500, 20, 100000, 0, -1.0)])


def simsearch_chain_case():
    """The reference's whole `simsearch -b` chain (max_mean -> calc -> write, oracle/reference_driver.run_simsearch_build)
    on the real-data scores of the simsearch_prep fixture: the index array, the bed text and, checked here, the oracle's
    restatement of the picks and of the text."""
    import tempfile
    from oracle import simsearch_oracle as sso
    g = np.load(HERE / "simsearch_prep_real_chr1_60k.npz")
    q, chrom, starts = g["scores_q"], g["chrom"], g["starts"]
    with tempfile.TemporaryDirectory() as tmp:
        path = Path(tmp) / "scores_x.txt.gz"
        with gzip.open(path, "wt", compresslevel=1) as f:
            f.write("".join("%s\t%d\t%d\t%s\n" % (chrom[i], starts[i], starts[i] + 200, "\t".join("%.5f" % (v / 1e5) for v in q[i]))
                            for i in range(len(q))))
        r = ref.run_simsearch_build(path, 125, 5, 25000, -1, -1.0, 100, n_jobs=3)
    idx = r["indices"]
    print("chain: regions", idx.shape, "matches per region (min/median/max)", [(int(f((idx > 0).sum(axis=1)))) for f in (np.min, np.median, np.max)],
          "leftovers", r["leftovers"])
    # oracle restatements against the reference, before the fixture is trusted
    coords = np.empty((len(q), 3), dtype=object)
    coords[:, 0], coords[:, 1], coords[:, 2] = chrom, starts.tolist(), (starts + 200).tolist()
    assert sso.bed_text(idx, coords, r["cube_coords"], 125, 5) == r["bed_text"], "bed text restatement"
    mism = 0
    for i in range(len(idx)):
        s0 = int(np.flatnonzero(starts == r["cube_coords"][i][1])[0]) // 5
        got = sso.similar_regions(r["reduced_genome"], r["cube_scores"][i], s0, 100)
        mism += int(not np.array_equal(got, idx[i]))
    print("chain: oracle picks differ from the reference for", mism, "of", len(idx), "regions (exact distance ties)")
    np.savez_compressed(HERE / "simsearch_chain_real_chr1_60k.npz", indices=idx, bed_digest=text_digest(r["bed_text"]),
                        bed_head=np.frombuffer(r["bed_text"][:2000], dtype=np.uint8), bed_bytes=np.int64(len(r["bed_text"])),
                        leftovers=np.array(r["leftovers"]), oracle_mismatches=np.int64(mism))


def roi_cases():
    """helpers.maxMean of the reference (the ROI selector that consumes the single-mode scores) on
    (a) S1 scores of a 200 000-bin real-data slice, window 50, and (b) two short synthetic chromosomes with odd /
    even windows.  Scores are the oracle's (bit-identical to the reference's, see test_oracle_golden)."""
    import warnings
    ref._import_reference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from epilogos.helpers import maxMean
    x = real_slice(100000, 200000)
    exp, scores = orc.expected_and_scores(x, 18, 1)
    n = len(scores)
    loc = np.empty((n, 3), dtype=object)
    loc[:, 0] = "chr1"; loc[:, 1] = np.arange(n) * 200; loc[:, 2] = np.arange(n) * 200 + 200
    rois, idx = maxMean(np.concatenate((loc, scores.sum(axis=1).reshape(n, 1)), axis=1), 50, 100)
    np.savez_compressed(HERE / "roi_real10_w50.npz", x=x.astype(np.int8), exp=exp, window=np.int64(50),
                        original_idx=idx.astype(np.int64), start=rois["Start"].to_numpy(np.int64),
                        end=rois["End"].to_numpy(np.int64), rolling_max=rois["RollingMax"].to_numpy(np.float64),
                        rolling_mean=rois["RollingMean"].to_numpy(np.float64))
    print("wrote roi_real10_w50", len(idx))
    rng = np.random.default_rng(17)
    for window in (50, 125, 7):
        n1, n2 = 3100, 2400
        sc = (rng.standard_normal((n1 + n2, 15)) * rng.choice([0.0, 0.2, 1.0], size=(n1 + n2, 1))).astype(np.float32)
        loc = np.empty((n1 + n2, 3), dtype=object)
        loc[:n1, 0] = "chr1"; loc[n1:, 0] = "chr2"
        st = np.concatenate([np.arange(n1), np.arange(n2)]) * 200
        loc[:, 1] = st; loc[:, 2] = st + 200
        rois, idx = maxMean(np.concatenate((loc, sc.sum(axis=1).reshape(-1, 1)), axis=1), window, 100)
        np.savez_compressed(HERE / ("roi_synth_w%d.npz" % window), scores=sc, starts=st.astype(np.int64),
                            chrom_split=np.int64(n1), window=np.int64(window), original_idx=idx.astype(np.int64),
                            start=rois["Start"].to_numpy(np.int64), end=rois["End"].to_numpy(np.int64),
                            rolling_max=rois["RollingMax"].to_numpy(np.float64),
                            rolling_mean=rois["RollingMean"].to_numpy(np.float64))
        print("wrote roi_synth_w%d" % window, len(idx))


def main():
    which = set(sys.argv[1:])

    def want(n):
        return not which or n in which

    real = real_slice()
    if want("real10"):
        single_case("real10_chr1_k18", real, 18, (1, 2, 3))
    if want("real10_mp"):
        # three worker processes: exercises splitRows chunking (helpers.py:102-120); results must not change
        single_case("real10_chr1_k18_nproc3", real[:1000], 18, (1, 2), keep_text=False, nproc=3)
    if want("synth833"):
        single_case("synth_c833_k18", orc.synth_states(1500, 833, 18, seed=1), 18, (1, 2), keep_text=False)
    if want("synth833u"):
        single_case("synth_uniform_c833_k18", orc.synth_states(600, 833, 18, seed=2, kind="uniform"), 18, (1, 2),
                    keep_text=False)
    if want("synth127"):
        single_case("synth_c127_k15", orc.synth_states(2000, 127, 15, seed=3), 15, (1, 2), keep_text=False)
    if want("s3small"):
        single_case("synth_s3_c12_k15", orc.synth_states(300, 12, 15, seed=4, kind="uniform"), 15, (3,),
                    keep_text=False)
        single_case("synth_s3_c40_k18", orc.synth_states(500, 40, 18, seed=5), 18, (3,), keep_text=False)
    if want("paired_real"):
        paired_case("paired_real10_k18", real[:, :5], real[:, 5:], 18, (1, 2), seed=7)
    if want("paired_synth"):
        xa = orc.synth_states(1200, 30, 18, seed=8)
        xb = orc.synth_states(1200, 25, 18, seed=9)
        paired_case("paired_synth_c30_c25_k18", xa, xb, 18, (1, 2), seed=10)
        paired_case("paired_synth_g20_k18", xa, xb, 18, (1, 2), seed=12, group_size=20)
        paired_case("paired_synth_q0_k18", xa[:400], xb[:400], 18, (1,), seed=13, quiescent_state=-1)
    if want("paired_gwide"):
        # -g larger than half the combined width: the second shuffled slice [:, G:2G] is clipped to N - G columns
        xa = orc.synth_states(400, 30, 18, seed=8)
        xb = orc.synth_states(400, 25, 18, seed=9)
        paired_case("paired_synth_g40_k18", xa, xb, 18, (1, 2), seed=14, group_size=40)
    if want("s3big"):
        s3_big_case("synth_s3_c833_k18")
    if want("roi"):
        roi_cases()
    if want("roi_wide"):
        roi_wide_case()
    if want("real_full"):
        real_full_case()
    if want("simsearch"):
        simsearch_case()
    if want("simsearch_prep"):
        simsearch_prep_case()
    if want("simsearch_chain"):
        simsearch_chain_case()


if __name__ == "__main__":
    main()
