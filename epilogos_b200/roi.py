"""Step 4 (single mode) -- regions of interest.  Mirror of the reference's roiSingle.py.

    main(outputDir, stateInfo, fileTag, expFreqPath, roiWidth, verbose)                     (roiSingle.py:10)

Reads the score stage's results (every `temp_scores_*.npz`, or what the score stage of this process handed over in
memory: epilogos_b200.handoff), orders the chromosomes (helpers.orderChromosomes, helpers.py:224-250), selects the
top 100 non-overlapping windows with the max-mean rule (native epi_roi_maxmean), names the strongest state of each
window, writes `regionsOfInterest_<tag>.txt` and removes the temp score files and the expected-frequency file exactly
as the reference does (roiSingle.py:40, 73-74).
"""
import ctypes
from os import remove
from pathlib import Path
from sys import argv

import numpy as np

from . import _lib, handoff
from .helpers import strToBool
from .run import getStateNames


def orderChromosomes(chromosomes):
    """Numbered chromosomes ascending, then the rest alphabetically (helpers.py:224-250)."""
    nums, names = [], []
    for c in chromosomes:
        tail = c.split("chr")[-1]
        (nums if tail.isdigit() or (tail.startswith("-") and tail[1:].isdigit()) else names).append(tail)
    return ["chr" + str(v) for v in sorted(int(t) for t in nums)] + ["chr" + t for t in sorted(names)]


def max_mean(starts, ends, score, window, max_regions=100):
    """helpers.maxMean on plain arrays; returns dict(original_idx, start, end, rolling_max, rolling_mean)."""
    score = np.ascontiguousarray(score, dtype=np.float64)
    starts = np.ascontiguousarray(starts, dtype=np.int64)
    ends = np.ascontiguousarray(ends, dtype=np.int64)
    out_i = np.empty(max_regions, dtype=np.int64)
    out_s = np.empty(max_regions, dtype=np.int64)
    out_e = np.empty(max_regions, dtype=np.int64)
    out_mx = np.empty(max_regions, dtype=np.float64)
    out_mn = np.empty(max_regions, dtype=np.float64)
    n_out = ctypes.c_int32(0)
    p = lambda a: ctypes.c_void_p(a.ctypes.data)
    _lib.call("epi_roi_maxmean", p(score), p(starts), p(ends), len(score), int(window), int(max_regions), p(out_i),
              p(out_s), p(out_e), p(out_mx), p(out_mn), ctypes.byref(n_out))
    k = n_out.value
    return dict(original_idx=out_i[:k], start=out_s[:k], end=out_e[:k], rolling_max=out_mx[:k], rolling_mean=out_mn[:k])


def permutation_pvalues(be, chunks, mismatch):
    """(k uint32, p, BH) over the bins of all chunks, or None when the score stage counted no permutations: k of the P
    shuffles of a bin whose statistic is at least the bin's, p = (1 + k) / (P + 1), and the Benjamini-Hochberg adjustment
    over all bins.  Chunks that disagree on P raise ValueError("<mismatch> on the number of permutations (...)")."""
    perms = {c.get("permutations") for c in chunks}
    if perms == {None}:
        return None
    if None in perms or len(perms) != 1:
        raise ValueError("{} on the number of permutations ({})".format(mismatch, sorted(str(p) for p in perms)))
    P = perms.pop()
    k = np.concatenate([np.asarray(c["exceedances"], dtype=np.uint32) for c in chunks])
    p = (k.astype(np.float64) + 1.0) / (P + 1.0)
    return k, p, be.bh_adjust(be.to_device(p)).cpu().numpy()


def readInData(outputDirPath, fileTag):
    """The score stage's results in chromosome order -> (chrom per row, starts, ends, scoreArr); temp files removed."""
    chunks = handoff.collect("scores", outputDirPath, fileTag)
    handoff.remove_temps("scores", outputDirPath, fileTag)
    return tuple(np.concatenate([c[k] for c in chunks]) for k in ("chrom", "start", "end", "scoreArr"))


def createTopScoresTxt(filePath, chrom, starts, ends, scoreArr, nameArr, roiWidth):
    """regionsOfInterest*.txt: chromosome, start, end, strongest state, |score| (5 decimals), sign (roiSingle.py:95-142).
    The ranking input is scoreArr.sum(axis=1) in float32 (roiSingle.py:118)."""
    sel = max_mean(starts, ends, scoreArr.sum(axis=1), roiWidth, 100)
    half = roiWidth // 2
    k = scoreArr.shape[1]
    lines = []
    for i, idx in enumerate(sel["original_idx"]):
        lo, hi = idx - half, idx + half + (1 if roiWidth % 2 else 0)
        col_max = scoreArr[lo:hi].max(axis=0)
        state = k - int(np.argmax(col_max[::-1]))              # ties -> the higher numbered state (roiSingle.py:125-129)
        s32 = float(np.float32(sel["rolling_max"][i]))
        lines.append("%s\t%d\t%d\t%s\t%.5f\t%s\n" % (chrom[idx], sel["start"][i], sel["end"][i], nameArr[state - 1],
                                                     abs(s32), "+" if s32 >= 0 else "-"))
    with open(filePath, "w") as out:
        out.write("".join(lines))


def main(outputDir, stateInfo, fileTag, expFreqPath, roiWidth, verbose):
    outputDirPath = Path(outputDir)
    names = getStateNames(stateInfo)
    if not verbose:
        print("    Reading in files\t", end="", flush=True)
    chrom, starts, ends, scoreArr = readInData(outputDirPath, fileTag)
    if not verbose:
        print("\t[Done]\n    Regions of interest txt\t", end="", flush=True)
    createTopScoresTxt(outputDirPath / "regionsOfInterest_{}.txt".format(fileTag), chrom, starts, ends, scoreArr, names,
                       roiWidth)
    if not verbose:
        print("\t[Done]", flush=True)
    remove(Path(expFreqPath))


if __name__ == "__main__":
    main(argv[1], argv[2], argv[3], argv[4], int(argv[5]), strToBool(argv[6]))
