"""Drive the UNMODIFIED reference (meuleman/epilogos, a checkout named by EPILOGOS_REFERENCE) on small inputs.

TEST / BENCHMARK INFRASTRUCTURE ONLY.  This file is the only place that imports the reference.  It exists to
(1) generate the golden fixtures committed under tests/golden/ (see tests/golden/make_golden.py),
(2) cross-check the numpy restatement in oracle/epilogos_oracle.py while authoring, and
(3) time the reference's own CPU path for bench.py's `--impl reference` arm and `cpu_baseline` leg.
Where no checkout is named, the package is imported from the byte-compiled copy oracle/_ref/ when one was staged
(oracle/stage_reference.py, git-ignored).  smoke() never imports this module, and the tests that compare against the
committed fixtures do not need it.

The reference cannot be imported as-is in this image: helpers.py:7 pulls in filter_regions.py which
imports natsort/pyranges (filter_regions.py:10), and run.py:14 pulls matplotlib/statsmodels.  None of
those modules is touched by the hot path (expected.py, expectedCombination.py, scores.py), so empty
stand-ins are registered in sys.modules before the import (SURVEY.md Appendix B).
"""
import sys
import types
import tempfile
from pathlib import Path

import numpy as np

from .stage_reference import staged_root

REFERENCE_ROOT = staged_root()

_STUBS = ["natsort", "pyranges", "matplotlib", "matplotlib.pyplot", "matplotlib.lines", "statsmodels",
          "statsmodels.stats", "statsmodels.stats.multitest", "pysam"]


def available():
    return REFERENCE_ROOT is not None


def _import_reference():
    for name in _STUBS:
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["statsmodels.stats.multitest"].multipletests = None
    sys.modules["matplotlib.lines"].Line2D = None
    if str(REFERENCE_ROOT) not in sys.path:
        sys.path.insert(0, str(REFERENCE_ROOT))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from epilogos.expected import main as expected_main                      # expected.py:11
        from epilogos.expectedCombination import main as combination_main        # expectedCombination.py:9
        from epilogos.scores import main as scores_main                          # scores.py:14
    return expected_main, combination_main, scores_main


def write_matrix_tsv(path, states1, chrom="chr1", bin_size=200, start_bin=0):
    """Write a 1-based state matrix in the reference's input format (README.md:286-292)."""
    states1 = np.asarray(states1)
    with open(path, "w") as f:
        for r in range(states1.shape[0]):
            lo = (start_bin + r) * bin_size
            f.write("%s\t%d\t%d\t" % (chrom, lo, lo + bin_size))
            f.write("\t".join(str(int(v)) for v in states1[r]))
            f.write("\n")


def run_single(states0, num_states, saliency, nproc=1, chrom="chr1"):
    """states0: 0-based [bins, C].  Returns dict(counts=int64 table, exp=float32 table, scores=f32 [bins,K],
    scores_text=bytes of the decompressed scores_*.txt.gz)."""
    import gzip
    expected_main, combination_main, scores_main = _import_reference()
    with tempfile.TemporaryDirectory() as d:
        d = Path(d)
        inp = d / "in"
        out = d / "out"
        inp.mkdir(); out.mkdir()
        f = inp / ("epilogos_matrix_%s.txt" % chrom)
        write_matrix_tsv(f, np.asarray(states0) + 1, chrom=chrom)
        tag = "in_s%d" % saliency
        expected_main(f, "null", num_states, saliency, out, tag, nproc, False)
        tmp = out / ("temp_exp_freq_%s_%s.npy" % (tag, f.name.split(".")[0]))
        counts = np.load(tmp)
        exp_path = out / ("exp_freq_%s.npy" % tag)
        combination_main(out, exp_path, tag, False)
        exp = np.load(exp_path)
        scores_main(f, "null", num_states, saliency, out, exp_path, tag, nproc, num_states - 1, -1, False)
        npz = np.load(out / ("temp_scores_%s_%s.npz" % (tag, f.name.split(".")[0])), allow_pickle=True)
        with gzip.open(out / ("scores_%s_%s.txt.gz" % (tag, f.name.split(".")[0])), "rb") as g:
            text = g.read()
        return dict(counts=counts, exp=exp, scores=np.array(npz["scoreArr"]), scores_text=text)


def run_paired(statesA0, statesB0, num_states, saliency, seed, quiescent_state=None, group_size=-1, nproc=1,
               chrom="chr1"):
    """Paired mode with a seeded parent RNG (np.random.seed(seed) before scores.main makes the unseeded
    shuffle of helpers.py:183-184 reproducible; SURVEY.md section 8a)."""
    import gzip
    expected_main, combination_main, scores_main = _import_reference()
    if quiescent_state is None:
        quiescent_state = num_states - 1
    with tempfile.TemporaryDirectory() as d:
        d = Path(d)
        a = d / "a"; b = d / "b"; out = d / "out"
        a.mkdir(); b.mkdir(); out.mkdir()
        fa = a / ("epilogos_matrix_%s.txt" % chrom)
        fb = b / ("epilogos_matrix_%s.txt" % chrom)
        write_matrix_tsv(fa, np.asarray(statesA0) + 1, chrom=chrom)
        write_matrix_tsv(fb, np.asarray(statesB0) + 1, chrom=chrom)
        tag = "a_b_s%d" % saliency
        stem = fa.name.split(".")[0]
        expected_main(fa, fb, num_states, saliency, out, tag, nproc, False)
        counts = np.load(out / ("temp_exp_freq_%s_%s.npy" % (tag, stem)))
        exp_path = out / ("exp_freq_%s.npy" % tag)
        combination_main(out, exp_path, tag, False)
        exp = np.load(exp_path)
        np.random.seed(seed)
        scores_main(fa, fb, num_states, saliency, out, exp_path, tag, nproc, quiescent_state, group_size, False)
        null = np.load(out / ("temp_nullDistances_%s_%s.npz" % (tag, stem)))["nullDistances"]
        quies = np.load(out / ("temp_quiescence_%s_%s.npz" % (tag, stem)))["quiescenceArr"]
        with gzip.open(out / ("pairwiseDelta_%s_%s.txt.gz" % (tag, stem)), "rb") as g:
            text = g.read()
        return dict(counts=counts, exp=exp, null_distances=np.array(null), quiescence=np.array(quies),
                    delta_text=text)


def simsearch_coords(nbins, chrom_split=None):
    """Coordinates of the non-reduced genome of the similarity-search fixtures: one chromosome, or chr1 = the first
    `chrom_split` bins and chr2 the rest (coordinates restart at 0 on chr2, so a start alone does not identify a bin)."""
    if chrom_split is None:
        return np.array(["chr1"] * nbins, dtype=object), np.arange(nbins, dtype=np.int64) * 200
    chrom = np.array(["chr1"] * chrom_split + ["chr2"] * (nbins - chrom_split), dtype=object)
    start = np.concatenate((np.arange(chrom_split), np.arange(nbins - chrom_split))).astype(np.int64) * 200
    return chrom, start


def run_simsearch(reduced_genome, roi_starts, window_bins, block_size, n_desired, chrom_split=None):
    """similaritySearch_calc.runEuclideanDistance (similaritySearch_calc.py:67-123) of the unmodified reference on an
    in-memory reduced genome; the ROIs are the windows of the genome that start at reduced bins `roi_starts`.
    Returns the int32 [len(roi_starts), n_desired] array the reference stores in simsearch_indices_*.npy."""
    import warnings
    import pandas as pd
    _import_reference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from epilogos import similaritySearch_calc as ssc
    reduced_genome = np.asarray(reduced_genome)
    g = len(reduced_genome)
    n_super = window_bins // block_size
    nbins = g * block_size
    chrom, start = simsearch_coords(nbins, chrom_split)
    genome_coords = pd.DataFrame({"Chromosome": chrom, "Start": start, "End": start + 200})
    roi_cube = np.stack([reduced_genome[s:s + n_super] for s in roi_starts])
    rows = [int(s) * block_size for s in roi_starts]
    roi_coords = pd.DataFrame({"Chromosome": [chrom[r] for r in rows], "Start": [int(start[r]) for r in rows],
                               "End": [int(start[r]) + window_bins * 200 for r in rows]})
    out = np.zeros((len(roi_starts), n_desired), dtype=np.int32)
    ssc._initEuclideanDistance(genome_coords, reduced_genome, roi_coords, roi_cube, out, window_bins, block_size, n_desired)
    ssc.runEuclideanDistance((0, len(roi_starts)))
    return out


def run_simsearch_prep(scores_path, window_bins, block_size, window_bp, filter_state, filter_score):
    """similaritySearch_max_mean.main (similaritySearch_max_mean.py:9-48) of the unmodified reference on a score file.
    Returns dict(genome_scores, genome_coords, cube_scores, cube_coords, reduced_genome) = the contents of
    genome_stats.npz, simsearch_cube.npz and reduced_genome.npy."""
    import contextlib
    import io
    import warnings
    _import_reference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from epilogos import similaritySearch_max_mean as mm
        with tempfile.TemporaryDirectory() as tmp:
            out = Path(tmp)
            with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                mm.main(out, Path(scores_path), int(window_bins), int(block_size), int(window_bp), int(filter_state),
                        float(filter_score))
            stats = np.load(out / "genome_stats.npz", allow_pickle=True)
            cube = np.load(out / "simsearch_cube.npz", allow_pickle=True)
            return dict(genome_scores=stats["scores"], genome_coords=stats["coords"], cube_scores=cube["scores"],
                        cube_coords=cube["coords"], reduced_genome=np.load(out / "reduced_genome.npy", allow_pickle=True))


def run_simsearch_build(scores_path, window_bins, block_size, window_bp, filter_state, filter_score, n_desired, n_jobs=1):
    """The reference's whole `simsearch -b` chain without SLURM: similaritySearch_max_mean.main ->
    similaritySearch_calc.main (one call per job, nCores = 1) -> similaritySearch_write.main.
    pysam is absent from this image and the writer puts its temporary file into the (read-only) reference tree, so two
    stand-ins are installed around the UNMODIFIED writer code: `pysam.tabix_compress` = a plain gzip copy and
    `pysam.tabix_index` = a placeholder file; `tempfile` is redirected to the output directory.  The bed TEXT is the
    reference's own.  Returns dict(indices int32 [regions, n_desired], bed_text bytes, cube_coords, cube_scores,
    reduced_genome)."""
    import contextlib
    import gzip
    import io
    import shutil
    import warnings
    _import_reference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from epilogos import similaritySearch_max_mean as mm
        from epilogos import similaritySearch_calc as ssc
        from epilogos import similaritySearch_write as ssw
        with tempfile.TemporaryDirectory() as tmp:
            out = Path(tmp) / "out"
            out.mkdir()

            def tabix_compress(src, dst, force=False):
                with open(src, "rb") as a, gzip.open(dst, "wb") as b:
                    shutil.copyfileobj(a, b)

            def tabix_index(fn, force=False, zerobased=False, preset=None):
                Path(str(fn) + ".tbi").write_bytes(b"placeholder")

            class _Tempfile:
                @staticmethod
                def NamedTemporaryFile(mode="w+b", delete=True, dir=None):
                    return tempfile.NamedTemporaryFile(mode=mode, delete=delete, dir=tmp)

            ssw.pysam.tabix_compress = tabix_compress
            ssw.pysam.tabix_index = tabix_index
            ssw.tempfile = _Tempfile
            with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                mm.main(out, Path(scores_path), int(window_bins), int(block_size), int(window_bp), int(filter_state),
                        float(filter_score))
                cube = np.load(out / "simsearch_cube.npz", allow_pickle=True)
                cube_scores, cube_coords = cube["scores"], cube["coords"]
                reduced = np.load(out / "reduced_genome.npy", allow_pickle=True)
                for tag in range(n_jobs):
                    ssc.main(out, int(window_bins), int(block_size), 1, int(n_desired), int(n_jobs), tag)
                ssw.main(out, int(window_bins), int(block_size), int(n_jobs), int(n_desired))
            with gzip.open(out / "simsearch.bed.gz", "rb") as f:
                bed = f.read()
            return dict(indices=np.load(out / "simsearch_indices.npy", allow_pickle=True), bed_text=bed,
                        cube_coords=cube_coords, cube_scores=cube_scores, reduced_genome=reduced,
                        leftovers=sorted(p.name for p in out.iterdir()))


# ------------------------------------------------------------------------------------------------
# timing of the reference's own `epilogos -l` compute stages (bench.py --impl reference / cpu_baseline)
# ------------------------------------------------------------------------------------------------
def write_matrix_tsv_gz(path, states0, chrom="chr1", bin_size=200, level=1):
    """Fast writer of the reference's input format (README.md:286-292) for benchmark samples: 0-based int labels ->
    1-based decimal text, one row per bin, gzip.  Vectorised (the per-row Python writer above takes minutes at
    100,000 x 833)."""
    import gzip
    v = np.asarray(states0).astype(np.int16) + 1
    rows, cols = v.shape
    cell = np.empty((rows, cols, 3), dtype=np.uint8)
    cell[..., 0] = 9                                   # tab
    cell[..., 1] = 48 + v // 10
    cell[..., 2] = 48 + v % 10
    keep = np.ones((rows, cols, 3), dtype=bool)
    keep[..., 1] = v >= 10                             # no leading zero
    flat = cell[keep]
    lens = keep.reshape(rows, -1).sum(axis=1)
    ends = np.cumsum(lens)
    with gzip.open(path, "wb", compresslevel=level) as f:
        lo = 0
        for r in range(rows):
            f.write(b"%s\t%d\t%d" % (chrom.encode(), r * bin_size, (r + 1) * bin_size))
            f.write(flat[lo:ends[r]].tobytes())
            f.write(b"\n")
            lo = ends[r]


def _parse_verbose_times(text):
    """Seconds the first worker spent in the compute loops, from the reference's own verbose timers
    (expected.py:108-114 / 141-160 / 187-202, scores.py:305-324 / 400-423 / 484-506): the `    Time:` line that
    follows `Calculating expected frequencies...` / `Calculating Scores...`."""
    total, armed = 0.0, False
    for line in text.splitlines():
        if line.startswith("Calculating expected frequencies") or line.startswith("Calculating Scores"):
            armed = True
        elif armed and line.strip().startswith("Time:"):
            try:
                total += float(line.split("Time:")[1])
            except ValueError:
                pass
            armed = False
    return total


def time_pipeline(file1, file2, num_states, saliency, nproc, workdir, verbose_timers=False):
    """expected.main -> expectedCombination.main -> scores.main of the unmodified reference on TSV(.gz) input file(s)
    with `nproc` worker processes (run.py:196/214, 231, 246/268 -- what `epilogos -l -c nproc` runs before the ROI step).
    Returns (seconds wall clock incl. parse + gz write, seconds of the first worker's compute loops or None)."""
    import os
    import time
    expected_main, combination_main, scores_main = _import_reference()
    out = Path(workdir) / "out"
    if out.exists():
        import shutil
        shutil.rmtree(out)
    out.mkdir(parents=True)
    tag = "bench_s%d" % saliency
    exp_path = out / ("exp_freq_%s.npy" % tag)
    log = Path(workdir) / "stdout.log"
    sys.stdout.flush()
    saved = os.dup(1)
    fd = os.open(str(log), os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    os.dup2(fd, 1)                                    # forked pool workers inherit it: their timers land in the log
    try:
        t0 = time.perf_counter()
        expected_main(file1, file2, num_states, saliency, out, tag, nproc, verbose_timers)
        combination_main(out, exp_path, tag, verbose_timers)
        scores_main(file1, file2, num_states, saliency, out, exp_path, tag, nproc, num_states - 1, -1, verbose_timers)
        sys.stdout.flush()
        wall = time.perf_counter() - t0
    finally:
        os.dup2(saved, 1)
        os.close(saved)
        os.close(fd)
    compute = _parse_verbose_times(log.read_text()) if verbose_timers else None
    return wall, compute
