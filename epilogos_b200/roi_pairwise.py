"""Step 4 (paired mode) -- null-distribution fit, p-values, pairwiseMetrics and regions of interest.  The statistics of
the reference's roiAndVisualPairwise.py (:177-242, 339-354), without its figures.

    main(outputDir, stateInfo, fileTag, expFreqPath, roiWidth, pval, numTrials, samplingSize, diagnostic, verbose)
    python -m epilogos_b200.roi_pairwise OUTPUT_DIR STATE_INFO FILE_TAG EXP_FREQ_PATH ROI_WIDTH PVAL \\
                                         [NUM_TRIALS SAMPLING_SIZE DIAGNOSTIC VERBOSE]

Inputs per chromosome: the distance (sum_s d^2 * sign(sum_s d) of the delta row after its "%.5f" text round trip) and
the max-difference state of every bin, the null distances and the quiescence mask.  They come from the score stage of
this process (session.handover: already reduced on the device) or from its files: pairwiseDelta_<tag>_<file>.txt.gz,
temp_nullDistances_<tag>_<file>.npz and temp_quiescence_<tag>_<file>.npz.  Both routes give the same bits.

With -n (`pval`):
  1. the null pool = the null distances of the non-quiescent bins of every file in chromosome order (every permutation);
  2. numTrials subsamples of samplingSize distinct pool entries (the whole pool once when it is not larger), drawn from
     a keyed permutation seeded by the run seed;
  3. scipy.stats.gennorm.fit of each subsample, on the device; the trial with the median NLL is kept;
  4. two-sided p-values of every bin's distance and their Benjamini-Hochberg adjustment over the genome.
With --roi-permutations P the score stage also found, per file, the P genome-wide maxima of the region null
(temp_regionNull_<tag>_<file>.npz or the hand-over; epilogos_b200.region_null): regionPermutation_<tag>.txt gives every
region of regionsOfInterest its family-wise p-value and regionNullMaxima_<tag>.npz keeps the maxima.
When the score stage counted null permutations (--null-permutations P: temp_permutations_<tag>_<file>.npz or the
hand-over), pairwisePermutation_<tag>.txt.gz holds per bin (chrom, start, end, k, p, BH): k of the P shuffles of the bin
whose |null distance| is at least |distance|, p = (1 + k) / (P + 1), and its Benjamini-Hochberg adjustment over all bins.
Outputs: pairwiseMetrics_<tag>.txt.gz (chrom, start, end, max-difference state, |distance|, sign[, p, BH]) and
regionsOfInterest_<tag>.txt (the 100 windows of largest max-mean |distance|; state and sign of the window's largest
|distance| bin[, its p and BH]).  Without -n the reference writes z-scores instead, whose definition is not available to
this package; the six-column files are written.  -d figures are not built (matplotlib is not a dependency).  The temp
files and exp_freq_<tag>.npy are removed, as the reference does (roiAndVisualPairwise.py:172, 343-344).
"""
import re
from os import remove
from pathlib import Path
from sys import argv

import numpy as np

from . import helpers, region_null, session, writer
from .helpers import strToBool
from .roi import max_mean, orderChromosomes, permutation_pvalues
from .run import getStateNames

STATS_SEED_SALT = "epilogos_b200 paired statistics: null subsamples"


def stats_seed(run_seed):
    """Seed of the null subsamples: the run seed (pairwise.run_seed) mixed with a constant, so that these draws are
    unrelated to the null shuffles drawn from the same run seed."""
    from .pairwise import file_seed
    return file_seed(run_seed, STATS_SEED_SALT)


def readInData(outputDirPath, fileTag, be):
    """{chrName: dict(distance, max_diff, null, quiescence, chrom, start, end)}: the score stage's hand-over for this
    directory, then the files of chromosomes not handed over."""
    chunks = {}
    for key in [k for k in session.handover if Path(k).parent == outputDirPath
                and Path(k).name.startswith("temp_nullDistances_{}_".format(fileTag))]:
        h = session.handover.pop(key)
        if "exceedances" in h:
            h["exceedances"] = h["exceedances"].cpu().numpy().view(np.uint32)
        chunks[h["chrName"]] = h
    nullFiles = sorted(outputDirPath.glob("temp_nullDistances_{}_*.npz".format(fileTag)))
    for nf in nullFiles:
        name = nf.name[len("temp_nullDistances_{}_".format(fileTag)):-len(".npz")]
        z = np.load(nf, allow_pickle=False)
        chrName = str(z["chrName"][0])
        if chrName in chunks:
            continue
        q = np.load(outputDirPath / "temp_quiescence_{}_{}.npz".format(fileTag, name), allow_pickle=False)
        loc, delta = helpers.read_scores(outputDirPath / "pairwiseDelta_{}_{}.txt.gz".format(fileTag, name))
        # the text already went through "%.5f": the reduction takes the parsed values as they are
        dist, md = be.pairwise_real_reduce(be.to_device(delta.astype(np.float32)), text_round_trip=False)
        chunks[chrName] = dict(chrName=chrName, distance=dist, max_diff=md,
                               null=be.to_device(np.ascontiguousarray(z["nullDistances"], dtype=np.float32)),
                               quiescence=be.to_device(q["quiescenceArr"].astype(np.uint8)),
                               chrom=loc["chrom"], start=loc["start"], end=loc["end"])
        pf = outputDirPath / "temp_permutations_{}_{}.npz".format(fileTag, name)
        if pf.exists():
            zp = np.load(pf, allow_pickle=False)
            chunks[chrName].update(exceedances=np.asarray(zp["exceedances"], dtype=np.uint32),
                                   permutations=int(zp["permutations"]))
    if not chunks:
        raise FileNotFoundError("no paired score-stage outputs (temp_nullDistances_{}_*.npz) in {}"
                                .format(fileTag, outputDirPath))
    order = orderChromosomes(list(chunks))
    return [chunks[c] for c in order]


def fit_null(be, chunks, numTrials, samplingSize, seed):
    """Steps 1-3 of the statistics: (beta, loc, scale, trial table).  The table has one row per trial run: beta, loc,
    scale, NLL, iterations, converged, and which trial was chosen."""
    import torch
    pool = torch.cat([be.null_pool(c["null"], c["quiescence"]).reshape(-1) for c in chunks])
    n = int(pool.numel())
    if n < 3:
        raise ValueError("the null distribution has {} non-quiescent values; fitting it needs at least 3".format(n))
    trials, size = (1, n) if n <= samplingSize else (numTrials, samplingSize)
    _, samples = be.null_subsample(pool, trials, size, seed)
    params, status = be.gennorm_fit(samples)
    params, status = np.asarray(params, dtype=np.float64), np.asarray(status)
    order = np.lexsort((np.arange(trials), params[:, 3]))       # NLL ascending, ties by trial index
    chosen = int(order[(trials - 1) // 2])
    table = dict(beta=params[:, 0], loc=params[:, 1], scale=params[:, 2], nll=params[:, 3],
                 iterations=status[:, 0].astype(np.int64), converged=status[:, 1].astype(bool), chosen=chosen,
                 pool_size=n, sample_size=size)
    return float(params[chosen, 0]), float(params[chosen, 1]), float(params[chosen, 2]), table


def roi_lines(chrom, starts, ends, distance, max_diff, names, roiWidth, pvals=None, bh=None):
    """regionsOfInterest text: max-mean windows of |distance|, state and sign of the window's largest |distance| bin."""
    absd = np.abs(distance.astype(np.float32))
    sel = max_mean(starts, ends, absd.astype(np.float64), roiWidth, 100)
    half = roiWidth // 2
    lines = []
    for i, idx in enumerate(sel["original_idx"]):
        lo, hi = idx - half, idx + half + (1 if roiWidth % 2 else 0)
        b = lo + int(np.argmax(absd[lo:hi]))
        line = "%s\t%d\t%d\t%s\t%.5f\t%s" % (chrom[idx], sel["start"][i], sel["end"][i], names[max_diff[b] - 1],
                                            float(np.float32(sel["rolling_max"][i])), "+" if distance[b] >= 0 else "-")
        if pvals is not None:
            line += "\t%.5e\t%.5e" % (pvals[b], bh[b])
        lines.append(line + "\n")
    return "".join(lines)


def main(outputDir, stateInfo, fileTag, expFreqPath, roiWidth, pval, numTrials=101, samplingSize=100000,
         diagnostic=False, verbose=False, backend=None, seed=None):
    """Returns dict(beta, loc, scale, trials) with -n (the chosen fit and the trial table), else None."""
    import torch
    outputDirPath = Path(outputDir)
    names = getStateNames(stateInfo)
    be = session.get_backend(backend)
    if not verbose:
        print("    Reading in files\t", end="", flush=True)
    chunks = readInData(outputDirPath, fileTag, be)
    distance_dev = torch.cat([c["distance"].reshape(-1) for c in chunks])
    distance = distance_dev.cpu().numpy()
    max_diff = torch.cat([c["max_diff"].reshape(-1) for c in chunks]).cpu().numpy().astype(np.int32)
    loc = dict(chrom=np.concatenate([np.asarray(c["chrom"], dtype=object) for c in chunks]),
               start=np.concatenate([np.asarray(c["start"], dtype=np.int64) for c in chunks]),
               end=np.concatenate([np.asarray(c["end"], dtype=np.int64) for c in chunks]))
    result = pvals = bh = None
    if pval:
        if not verbose:
            print("\t[Done]\n    Fitting the null distribution\t", end="", flush=True)
        if seed is None:
            from .pairwise import run_seed
            seed = run_seed()
        beta, fit_loc, scale, table = fit_null(be, chunks, numTrials, samplingSize, stats_seed(seed))
        if not verbose:
            print("\t[Done]\n    p-values\t", end="", flush=True)
        p_dev = be.gennorm_pvalues(distance_dev, beta, fit_loc, scale)
        bh = be.bh_adjust(p_dev).cpu().numpy()
        pvals = p_dev.cpu().numpy()
        result = dict(beta=beta, loc=fit_loc, scale=scale, trials=table)
    if not verbose:
        print("\t[Done]\n    Metrics and regions of interest\t", end="", flush=True)
    writer.write_metrics_text(outputDirPath / "pairwiseMetrics_{}.txt.gz".format(fileTag), loc, names, max_diff,
                              distance, pvals, bh)
    (outputDirPath / "regionsOfInterest_{}.txt".format(fileTag)).write_text(
        roi_lines(loc["chrom"], loc["start"], loc["end"], distance, max_diff, names, roiWidth, pvals, bh))
    # k = #{p < P : |null(b, p)| >= |distance(b)|}
    perm = permutation_pvalues(be, chunks, "temp_permutations files are missing for some chromosomes or disagree")
    if perm is not None:
        writer.write_permutations_text(outputDirPath / "pairwisePermutation_{}.txt.gz".format(fileTag), loc, *perm)
    # the region null (--roi-permutations): regionPermutation_<tag>.txt and regionNullMaxima_<tag>.npz
    region_null.read_temps(outputDirPath, fileTag, chunks)
    region = region_null.combine(chunks, "temp_regionNull files are missing for some chromosomes or disagree")
    if region is not None:
        region_null.write_outputs(outputDirPath, fileTag, loc["chrom"], loc["start"], loc["end"],
                                  np.abs(distance.astype(np.float32)), region)
    if not verbose:
        print("\t[Done]", flush=True)
    if diagnostic:
        print("    Diagnostic figures (-d) are not built: matplotlib is not a dependency of this package", flush=True)
    pattern = re.compile(r"^temp_(nullDistances|quiescence|permutations|regionNull)_{}_.*\.npz$".format(re.escape(fileTag)))
    for f in outputDirPath.iterdir():
        if pattern.match(f.name):
            remove(f)
    if Path(expFreqPath).exists():
        remove(Path(expFreqPath))
    return result


if __name__ == "__main__":
    extra = argv[7:]
    main(argv[1], argv[2], argv[3], argv[4], int(argv[5]), strToBool(argv[6]),
         int(extra[0]) if len(extra) > 0 else 101, int(extra[1]) if len(extra) > 1 else 100000,
         strToBool(extra[2]) if len(extra) > 2 else False, strToBool(extra[3]) if len(extra) > 3 else False)
