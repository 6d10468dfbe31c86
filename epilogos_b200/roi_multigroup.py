"""Step 4 (multi-group comparison, `--multigroup`) -- multigroupMetrics and regions of interest.

    main(outputDir, stateInfo, fileTag, expFreqPath, roiWidth, verbose)
    python -m epilogos_b200.roi_multigroup OUTPUT_DIR STATE_INFO FILE_TAG EXP_FREQ_PATH ROI_WIDTH

Inputs per chromosome, from the score stage of this process (epilogos_b200.handoff) or from
temp_multigroup_<tag>_<file>.npz (epilogos_b200.multigroup): the statistic T of every bin, the group g* and state s* that
drive it, the sign of S_g*[s*] - m[s*], and with --null-permutations P the count k of the P shuffles whose T is at least
as large.
Outputs, bins in chromosome order:
  multigroupMetrics_<tag>.txt.gz  chrom, start, end, "%.5e" T, group, state, +/- [, k, "%.5e" p, "%.5e" BH], with
                                  p = (1 + k) / (P + 1) and BH its Benjamini-Hochberg adjustment over all bins;
  regionsOfInterest_<tag>.txt     the 100 windows of largest max-mean T (epi_roi_maxmean): chrom, start, end, then group,
                                  state, sign and "%.5e" T of the window's first bin of largest T [, its p and BH].
With --roi-permutations P (temp_regionNull_<tag>_<file>.npz or the hand-over, epilogos_b200.region_null), also
  regionPermutation_<tag>.txt     per region of regionsOfInterest, in its order: chrom, start, end, "%.5e" window mean of
                                  T, k, "%.5e" family-wise p;
  regionNullMaxima_<tag>.npz      {maxima int64 [P], window, permutations}: the genome-wide maxima of the window sums.
The temp files and exp_freq_<tag>.npy are removed.
"""
from os import remove
from pathlib import Path
from sys import argv

import numpy as np

from . import handoff, region_null, session, writer
from .roi import max_mean, permutation_pvalues
from .run import getStateNames


def roi_lines(chrom, starts, ends, t, group, state, sign, group_names, state_names, roiWidth, pvals=None, bh=None):
    sel = max_mean(starts, ends, t, roiWidth, 100)
    half = roiWidth // 2
    lines = []
    for i, idx in enumerate(sel["original_idx"]):
        lo, hi = idx - half, idx + half + (1 if roiWidth % 2 else 0)
        b = max(lo, 0) + int(np.argmax(t[max(lo, 0):hi]))
        line = "%s\t%d\t%d\t%s\t%s\t%s\t%.5e" % (chrom[idx], sel["start"][i], sel["end"][i], group_names[group[b]],
                                                 state_names[state[b]], "-" if sign[b] < 0 else "+", t[b])
        if pvals is not None:
            line += "\t%.5e\t%.5e" % (pvals[b], bh[b])
        lines.append(line + "\n")
    return "".join(lines)


def main(outputDir, stateInfo, fileTag, expFreqPath, roiWidth, verbose=False, backend=None):
    outputDirPath = Path(outputDir)
    names = getStateNames(stateInfo)
    be = session.get_backend(backend)
    if not verbose:
        print("    Multi-group metrics and regions of interest\t", end="", flush=True)
    chunks = handoff.collect("multigroup", outputDirPath, fileTag)
    group_names = chunks[0]["groups"]
    cat = lambda key, dtype: np.concatenate([np.asarray(c[key], dtype=dtype) for c in chunks])   # noqa: E731
    loc = dict(chrom=cat("chrom", object), start=cat("start", np.int64), end=cat("end", np.int64))
    t, group, state, sign = cat("t", np.float64), cat("group", np.uint8), cat("state", np.uint8), cat("sign", np.int8)
    k, p, bh = permutation_pvalues(be, chunks, "temp_multigroup files disagree") or (None, None, None)
    writer.write_multigroup_text(outputDirPath / "multigroupMetrics_{}.txt.gz".format(fileTag), loc, t, group, state,
                                 sign, group_names, names, k, p, bh)
    (outputDirPath / "regionsOfInterest_{}.txt".format(fileTag)).write_text(
        roi_lines(loc["chrom"], loc["start"], loc["end"], t, group, state, sign, group_names, names, roiWidth, p, bh))
    region = region_null.combine(chunks, "temp_regionNull files are missing for some chromosomes or disagree")
    if region is not None:
        region_null.write_outputs(outputDirPath, fileTag, loc["chrom"], loc["start"], loc["end"], t, region)
    handoff.remove_temps("multigroup", outputDirPath, fileTag)
    if Path(expFreqPath).exists():
        remove(Path(expFreqPath))
    if not verbose:
        print("\t[Done]", flush=True)


if __name__ == "__main__":
    main(argv[1], argv[2], argv[3], argv[4], int(argv[5]))
