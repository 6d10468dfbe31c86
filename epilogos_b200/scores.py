"""Stage 3 -- per-bin KL scores.  Mirror of the reference's scores.py.

    main(file1, file2, numStates, saliency, outputDir, expFreqPath, fileTag, numProcesses, quiescentState,
         groupSize, verbose)                                                             (scores.py:14)

Single mode writes `scores_<tag>_<file>.txt.gz` and `temp_scores_<tag>_<file>.npz` (scores.py:163-169).
Rows are sharded over the ranks; each rank scores its own bins against the shared expected table and the
float32 rows are gathered on rank 0 for writing (the reference's workers write disjoint slices of a shared
RawArray, scores.py:142-157).
"""
from pathlib import Path
from sys import argv
from time import time

import numpy as np

from . import dist, helpers, session, writer


def main(file1, file2, numStates, saliency, outputDir, expFreqPath, fileTag, numProcesses, quiescentState, groupSize,
         verbose, backend=None, group=None, permutations=0, region_permutations=0, region_seed=None, roi_width=None):
    tTotal = time()
    file1Path, file2Path, outputDirPath = Path(file1), Path(file2), Path(outputDir)
    filename = file1Path.name.split(".")[0]
    if not verbose and dist.rank() == 0:
        print("    {}\t".format(filename), end="", flush=True)
    if group is not None and group.multi is not None:
        from .multigroup import calculateScoresMultigroup
        calculateScoresMultigroup(saliency, file1Path, numStates, outputDirPath, expFreqPath, fileTag, filename, verbose,
                                  backend, group=group, permutations=permutations,
                                  region_permutations=region_permutations, region_seed=region_seed, roi_width=roi_width)
    elif str(file2) == "null":
        calculateScores(saliency, file1Path, numStates, outputDirPath, expFreqPath, fileTag, filename, verbose,
                        backend, group=group)
    else:
        from .pairwise import calculateScoresPairwise
        calculateScoresPairwise(saliency, file1Path, file2Path, numStates, outputDirPath, expFreqPath, fileTag,
                                filename, quiescentState, groupSize, verbose, backend, group=group,
                                permutations=permutations, region_permutations=region_permutations,
                                region_seed=region_seed, roi_width=roi_width)
    if dist.rank() == 0:
        print("Total Time:", time() - tTotal, flush=True) if verbose else print("\t[Done]", flush=True)
    dist.barrier()


def calculateScores(saliency, file1Path, numStates, outputDirPath, expFreqPath, fileTag, filename, verbose,
                    backend=None, group=None):
    if saliency not in (1, 2, 3):
        raise ValueError("Please ensure that saliency metric is either 1, 2, or 3")
    be = session.get_backend(backend)
    shard = session.load_shard(file1Path, Path("null"), numStates, backend, group=group)
    exp = be.to_device(np.load(expFreqPath, allow_pickle=False))
    if saliency in (1, 2):
        local = be.scores(shard.counts(), shard.width, saliency, exp)
    else:
        local = be.scores_s3(shard.states_device(), shard.width, numStates, exp)
    scoreArr = dist.gather_rows(local, shard.total_rows)
    loc = _gather_locations(shard)
    if dist.rank() == 0:
        from . import timing
        with timing.stage("device -> host", sync_cuda=True):
            scoreArr = scoreArr.cpu().numpy()
        writer.write_scores_text(outputDirPath / "scores_{}_{}.txt.gz".format(fileTag, filename), scoreArr, loc)
        chrName = loc["chrom"][0] if len(loc["chrom"]) else ""
        npz = outputDirPath / "temp_scores_{}_{}.npz".format(fileTag, filename)
        import os
        if session.handover_enabled and not os.environ.get("EPILOGOS_B200_KEEP_TEMP"):
            # the ROI stage runs next, in this process: hand the arrays over in memory (session.handover)
            session.handover[str(npz)] = dict(chrName=str(chrName), scoreArr=scoreArr, chrom=loc["chrom"],
                                              start=np.asarray(loc["start"], dtype=np.int64),
                                              end=np.asarray(loc["end"], dtype=np.int64))
        else:
            helpers.savez_level(npz, chrName=np.array([chrName]), scoreArr=scoreArr, locationArr=writer.location_array(loc))


def _gather_locations(shard):
    """Locations of all rows on rank 0 (each rank parsed only its own row range)."""
    if dist.world_size() == 1:
        return shard.loc
    if shard.reader is not None:                 # the rows were dealt by one reader: rank 0 got every location with them
        return shard.loc_full if dist.rank() == 0 else None
    import torch.distributed as td
    parts = [None] * dist.world_size() if dist.rank() == 0 else None
    td.gather_object(shard.loc, parts, dst=0)
    if dist.rank() != 0:
        return None
    return {k: np.concatenate([p[k] for p in parts]) for k in ("chrom", "start", "end")}   # ids are per-rank: dropped


if __name__ == "__main__":
    main(argv[1], argv[2], int(argv[3]), int(argv[4]), argv[5], argv[6], argv[7], int(argv[8]), int(argv[9]),
         int(argv[10]), helpers.strToBool(argv[11]))
