"""Stage 1 -- per-file expected (background) COUNT tables.  Mirror of the reference's expected.py.

    main(file1, file2, numStates, saliency, outputDir, fileTag, numProcesses, verbose)      (expected.py:11)

Same arguments, same output file (`temp_exp_freq_<tag>_<file>.npy`, int64 counts, expected.py:220-223), same
ValueError for a saliency outside 1..3 (expected.py:80-81).  Rows are sharded over the torch.distributed
ranks (one GPU each) instead of a multiprocessing.Pool; the per-shard integer tables are summed with an
all-reduce (expected.py:85 does np.sum over the workers' results).  `numProcesses` is accepted for signature
compatibility: parallelism comes from the process group.
"""
from pathlib import Path
from sys import argv
from time import time

import numpy as np

from . import dist, helpers, session


def main(file1, file2, numStates, saliency, outputDir, fileTag, numProcesses, verbose, backend=None, group=None):
    tTotal = time()
    file1Path, file2Path, outputDirPath = Path(file1), Path(file2), Path(outputDir)
    filename = file1Path.name.split(".")[0]                                         # expected.py:31
    if saliency not in (1, 2, 3):
        raise ValueError("Please ensure that saliency metric is either 1, 2, or 3")
    if saliency == 3 and str(file2) != "null":
        raise ValueError("Please ensure that saliency metric is either 1 or 2 for Pairwise Epilogos")
    if not verbose and dist.rank() == 0:
        print("    {}\t".format(filename), end="", flush=True)

    shard = session.load_shard(file1Path, file2Path, numStates, backend, group=group)
    table = calculateExpected(saliency, shard, numStates, backend)
    if dist.rank() == 0:
        storeExpArray(table, outputDirPath, fileTag, filename)
        print("Total Time:", time() - tTotal, flush=True) if verbose else print("\t[Done]", flush=True)
    dist.barrier()


def calculateExpected(saliency, shard, numStates, backend=None):
    """Integer table of the whole file: per-rank table of the rank's rows, all-reduced (sum)."""
    be = session.get_backend(backend)
    if saliency in (1, 2):
        local = be.expected_table(shard.counts(), shard.width, saliency)
        dist.all_reduce_sum(local)
        return local.cpu().numpy().astype(np.int64, copy=False)
    # S3: the ranks all-reduce the int32 tile buffer of the one-hot Gram matrix (upper triangle only), then the
    # [C][C][K][K] int64 table (what np.sum over the workers' int32 tables yields, SURVEY.md 8a) is assembled
    tiles, plan = be.s3_tiles(shard.states_device(), shard.width, numStates)
    dist.all_reduce_sum(tiles)
    counts = be.s3_counts(tiles, plan, shard.width, numStates, shard.total_rows)
    return counts.cpu().numpy().astype(np.int64, copy=False)


def _rows_matrix(file1Path, file2Path, rowsToCalc, numStates):
    rows = (int(rowsToCalc[0]), int(rowsToCalc[1]))
    _, x = helpers.read_matrix(file1Path, rows, want_locations=False, num_states=numStates)
    if str(file2Path) != "null":
        _, xb = helpers.read_matrix(file2Path, rows, want_locations=False, num_states=numStates)
        x = np.concatenate((x, xb), axis=1)               # the union of both groups (helpers.py:173-179)
    return x


def s1Calc(file1Path, file2Path, rowsToCalc, numStates, verbose, backend=None):
    """The reference's per-chunk worker under its own name (expected.py:90-116): int64 [numStates] label counts of rows
    [rowsToCalc[0], rowsToCalc[1]) of the file (of both files side by side in paired mode), computed on the GPU."""
    be = session.get_backend(backend)
    x = _rows_matrix(file1Path, file2Path, rowsToCalc, numStates)
    return be.expected_table(be.counts(x, numStates), x.shape[1], 1).cpu().numpy().astype(np.int64, copy=False)


def s2Calc(file1Path, file2Path, rowsToCalc, numStates, verbose, backend=None):
    """expected.py:119-162: int64 [numStates, numStates] ordered-pair counts of the rows."""
    be = session.get_backend(backend)
    x = _rows_matrix(file1Path, file2Path, rowsToCalc, numStates)
    return be.expected_table(be.counts(x, numStates), x.shape[1], 2).cpu().numpy().astype(np.int64, copy=False)


def s3Calc(file1Path, rowsToCalc, numStates, verbose, backend=None):
    """expected.py:165-204: [C, C, numStates, numStates] counts of (biosample pair, state pair) over the rows (int32 in
    the reference's worker, summed to int64 by its caller; int64 here)."""
    be = session.get_backend(backend)
    x = _rows_matrix(file1Path, "null", rowsToCalc, numStates)
    tiles, plan = be.s3_tiles(be.states_to_device(x), x.shape[1], numStates)
    return be.s3_counts(tiles, plan, x.shape[1], numStates, x.shape[0]).cpu().numpy().astype(np.int64, copy=False)


def storeExpArray(expFreqArr, outputDirPath, fileTag, filename):
    expFreqPath = Path(outputDirPath) / "temp_exp_freq_{}_{}.npy".format(fileTag, filename)
    np.save(expFreqPath, expFreqArr, allow_pickle=False)


if __name__ == "__main__":
    main(argv[1], argv[2], int(argv[3]), int(argv[4]), argv[5], argv[6], int(argv[7]), helpers.strToBool(argv[8]))
