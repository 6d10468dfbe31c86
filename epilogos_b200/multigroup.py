"""Multi-group score stage (paired mode, `--groups ... --multigroup A,B,C`): one test per bin of whether G >= 2 disjoint
groups of biosamples differ.

Group g (n_g biosamples) is scored at its own width against the background of the union of the groups (the expected
table steps 1 and 2 make from the union's counts).  Per bin, CudaBackend.multigroup_stat gives the size-weighted
between-group sum of squares T of the score vectors, the group g* and state s* that drive it and the sign of
S_g*[s*] - m[s*] (include/epilogos_b200.h, csrc/multigroup.cu).  With --null-permutations P, k of P shuffles of the bin's
labels over the groups have a T at least as large (drawn on the device, keyed by the file seed, the permutation and the
GLOBAL bin, so the counts do not depend on the sharding).

Output (rank 0): the per-bin results go to step 4 in memory or to temp_multigroup_<tag>_<file>.npz
{chrName, groups, t float64, group uint8, state uint8, sign int8, chrom, start, end[, exceedances uint32, permutations]}.
"""
import numpy as np

from . import dist, handoff, region_null, session
from .pairwise import file_seed, run_seed
from .scores import _gather_locations


def calculateScoresMultigroup(saliency, file1Path, numStates, outputDirPath, expFreqPath, fileTag, filename, verbose,
                              backend=None, group=None, permutations=0, seed=None, region_permutations=0,
                              region_seed=None, roi_width=None, strata=None):
    """`region_permutations` P > 0: also the file's maxima of the region null over `region_seed`'s P label splits of the
    groups' columns (epilogos_b200.region_null), handed to step 4 or written to temp_regionNull_<tag>_<file>.npz.
    `strata` (groups.Strata, --strata): the permutations and the region splits shuffle labels only within strata."""
    if saliency not in (1, 2):
        raise ValueError("Please ensure that saliency metric is either 1 or 2 for Pairwise Epilogos")
    region_null.check_seed(region_permutations, region_seed)
    be = session.get_backend(backend)
    view = session.load_shard(file1Path, file1Path, numStates, backend, group=group)
    exp = be.to_device(np.load(expFreqPath, allow_pickle=False))
    cnt, sizes = view.group_blocks(), view.sizes
    by_strata = {}
    if strata is not None:
        from . import groups
        by_strata = {"strata": groups.stratify(view, strata)}
    t, g, s, sign = be.multigroup_stat(cnt, sizes, saliency, exp)
    exceed = None
    if permutations > 0:
        exceed = be.multigroup_exceedances(cnt, sizes, t, permutations, file_seed(run_seed(seed), filename), view.lo,
                                           saliency, exp, **by_strata)
    region = None
    if region_permutations > 0:
        cols = view.grouped()
        region = region_null.shard_maxima(be, "multigroup", cols.device_matrix(), cols.head, sizes, numStates, roi_width,
                                          region_permutations, region_seed, saliency, exp, **by_strata)
    total = view.total_rows
    t, g, s, sign = (dist.gather_rows(a, total) for a in (t, g, s, sign))
    loc = _gather_locations(view)
    extra = handoff.optional_parts(file1Path, loc, total, exceed, permutations, region, roi_width, region_permutations)
    if dist.rank() == 0:
        handoff.publish("multigroup", outputDirPath, fileTag, filename, handoff.record(
            loc, groups=np.asarray(group.multi, dtype=object), t=t.cpu().numpy(), group=g.cpu().numpy(),
            state=s.cpu().numpy(), sign=sign.cpu().numpy(), **extra))
