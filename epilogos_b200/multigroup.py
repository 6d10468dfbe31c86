"""Multi-group score stage (paired mode, `--groups ... --multigroup A,B,C`): one test per bin of whether G >= 2 disjoint
groups of biosamples differ.

Group g (n_g biosamples) is scored at its own width against the background of the union of the groups (the expected
table steps 1 and 2 make from the union's counts).  Per bin, CudaBackend.multigroup_stat gives the size-weighted
between-group sum of squares T of the score vectors, the group g* and state s* that drive it and the sign of
S_g*[s*] - m[s*] (include/epilogos_b200.h, csrc/multigroup.cu).  With --null-permutations P, k of P shuffles of the bin's
labels over the groups have a T at least as large (drawn on the device, keyed by the file seed, the permutation and the
GLOBAL bin, so the counts do not depend on the sharding).

Output (rank 0): the per-bin results go to step 4 in memory (session.handover) or to temp_multigroup_<tag>_<file>.npz
{chrName, groups, t float64, group uint8, state uint8, sign int8, chrom, start, end[, exceedances uint32, permutations]}.
"""
import os
from pathlib import Path

import numpy as np

from . import dist, helpers, session
from .pairwise import file_seed, run_seed
from .scores import _gather_locations


def calculateScoresMultigroup(saliency, file1Path, numStates, outputDirPath, expFreqPath, fileTag, filename, verbose,
                              backend=None, group=None, permutations=0, seed=None, region_permutations=0,
                              region_seed=None, roi_width=None):
    """`region_permutations` P > 0: also the file's maxima of the region null over `region_seed`'s P label splits of the
    groups' columns (epilogos_b200.region_null), handed to step 4 or written to temp_regionNull_<tag>_<file>.npz."""
    if saliency not in (1, 2):
        raise ValueError("Please ensure that saliency metric is either 1 or 2 for Pairwise Epilogos")
    if region_permutations > 0 and region_seed is None:
        raise ValueError("region permutations need the run's region seed (region_null.region_seed), drawn once per run")
    be = session.get_backend(backend)
    view = session.load_shard(file1Path, file1Path, numStates, backend, group=group)
    exp = be.to_device(np.load(expFreqPath, allow_pickle=False))
    cnt, sizes = view.group_blocks(), view.sizes
    t, g, s, sign = be.multigroup_stat(cnt, sizes, saliency, exp)
    exceed = None
    if permutations > 0:
        exceed = be.multigroup_exceedances(cnt, sizes, t, permutations, file_seed(run_seed(seed), filename), view.lo,
                                           saliency, exp)
    region = None
    if region_permutations > 0:
        from . import region_null
        cols = view.grouped()
        region = region_null.shard_maxima(be, "multigroup", cols.device_matrix(), cols.head, sizes, numStates, roi_width,
                                          region_permutations, region_seed, saliency, exp)
    total = view.total_rows
    t, g, s, sign = (dist.gather_rows(a, total) for a in (t, g, s, sign))
    if exceed is not None:
        exceed = dist.gather_rows(exceed, total)
    loc = _gather_locations(view)
    if dist.rank() != 0:
        return
    if region is not None:
        region_null.check_one_chromosome(loc["chrom"], file1Path)
    chrName = loc["chrom"][0] if len(loc["chrom"]) else ""
    out = dict(chrName=str(chrName), groups=list(group.multi), t=t.cpu().numpy(), group=g.cpu().numpy(),
               state=s.cpu().numpy(), sign=sign.cpu().numpy(), chrom=np.asarray(loc["chrom"], dtype=object),
               start=np.asarray(loc["start"], dtype=np.int64), end=np.asarray(loc["end"], dtype=np.int64))
    if exceed is not None:
        out.update(exceedances=exceed.cpu().numpy().view(np.uint32), permutations=int(permutations))
    path = Path(outputDirPath) / "temp_multigroup_{}_{}.npz".format(fileTag, filename)
    if session.handover_enabled and not os.environ.get("EPILOGOS_B200_KEEP_TEMP"):
        session.handover[str(path)] = out          # step 4 runs next, in this process
        if region is not None:
            region_null.stage_output(outputDirPath, fileTag, filename, chrName, region.cpu().numpy(), roi_width,
                                     region_permutations, out)
        return
    if region is not None:
        region_null.stage_output(Path(outputDirPath), fileTag, filename, chrName, region.cpu().numpy(), roi_width,
                                 region_permutations, None)
    extra = {} if exceed is None else dict(exceedances=out["exceedances"],
                                           permutations=np.array(int(permutations), dtype=np.int64))
    helpers.savez_level(path, chrName=np.array([chrName]), groups=np.array(out["groups"]), t=out["t"],
                        group=out["group"], state=out["state"], sign=out["sign"], chrom=out["chrom"].astype(str),
                        start=out["start"], end=out["end"], **extra)
