"""Paired-mode score stage.  Mirror of scores.calculateScoresPairwise (scores.py:172-256) and of the paired
branches of s1Score / s2Score (scores.py:282-303, 319-322, 373-398, 414-421).

Outputs (rank 0): `pairwiseDelta_<tag>_<file>.txt.gz`, `temp_nullDistances_<tag>_<file>.npz`
{chrName, nullDistances float32[B]}, `temp_quiescence_<tag>_<file>.npz` {chrName, quiescenceArr bool[B]}, and with
--null-permutations `temp_permutations_<tag>_<file>.npz` {chrName, exceedances uint32[B], permutations}.  When the
paired statistics stage (roi_pairwise) runs next in this process, the two temp files are not written: their content and
the reduced real deltas are handed over in memory (session.handover).

Null shuffles.  The reference shuffles each combined row once with the unseeded global numpy RNG
(helpers.py:183-184).  Two modes are provided (environment variable EPILOGOS_B200_NULL or the `null_mode`
argument):
  "reference" -- draw argsort(np.random.rand(rows, N)) on the host exactly as the reference does and replay
                 those indices on the GPU: bit-reproducible against a seeded single-process reference run.
  "device"    -- (default) draw the shuffle on the GPU from the per-bin counts with a counter-based Philox
                 stream; same distribution, no host RNG, supports `nperm` > 1 shuffles per bin.  The stream of a
                 bin is keyed by (run seed mixed with the file name, GLOBAL bin index, permutation): every file
                 and every bin gets its own independent draws (as in the reference, which draws fresh shuffles
                 for every file), and the result does not depend on how many GPUs share the rows.  The run seed
                 is `seed`, else $EPILOGOS_B200_SEED, else fresh entropy (the reference is unseeded).

In "reference" mode the S2 scores are evaluated term by term (EPI_SCORE_DIRECT: the reference's own float64
expression) so that delta text and null distances are byte-identical to a seeded reference run; the default
mode uses the tensor-core TABLE evaluation (within 1e-9 of it, float32 equal except rare 1-ulp cases).
"""
import hashlib
import os
from pathlib import Path

import numpy as np

from . import dist, helpers, session, writer
from .scores import _gather_locations


def run_seed(seed=None):
    """The 64-bit seed of this run's null draws: explicit argument, $EPILOGOS_B200_SEED, or fresh entropy drawn on
    rank 0 and shared with every rank (all ranks must key their bins with the same seed)."""
    if seed is None and os.environ.get("EPILOGOS_B200_SEED", "") != "":
        seed = int(os.environ["EPILOGOS_B200_SEED"])
    if seed is None:
        seed = int.from_bytes(os.urandom(8), "little")
        if dist.world_size() > 1:
            import torch.distributed as td
            box = [seed]
            td.broadcast_object_list(box, src=0)
            seed = box[0]
    return int(seed) & (2 ** 64 - 1)


def file_seed(seed, filename):
    """Run seed mixed with the input file's name: chromosomes draw from unrelated streams."""
    h = hashlib.blake2b(str(filename).encode(), digest_size=8, key=int(seed).to_bytes(8, "little")).digest()
    return int.from_bytes(h, "little")


def shuffled_widths(c1, c2, groupSize):
    """Widths of the two shuffled arrays readStates returns (helpers.py:190-194): the group widths, or with -g G the
    slices [:, :G] and [:, G:2G] of the N = c1 + c2 shuffled columns, which numpy clips to the array."""
    if groupSize == -1:
        return c1, c2
    n = c1 + c2
    return min(groupSize, n), max(0, min(groupSize, n - groupSize))


def calculateScoresPairwise(saliency, file1Path, file2Path, numStates, outputDirPath, expFreqPath, fileTag, filename,
                            quiescentState, groupSize, verbose, backend=None, null_mode=None, seed=None, nperm=1,
                            group=None, permutations=0, region_permutations=0, region_seed=None, roi_width=None):
    """`permutations` P > 0: also count, for every bin, how many of P device-drawn null shuffles (permutations 0..P-1 of
    the device sampler, scored like the run's null) are at least as far from 0 as the bin's real distance, and hand the
    counts to step 4 (session.handover) or write them to temp_permutations_<tag>_<file>.npz {chrName, exceedances
    uint32[B], permutations}.  Nothing else changes: in device mode permutation 0 is the run's own null.
    `region_permutations` P > 0: also the file's maxima of the region null over `region_seed`'s P label splits of the
    combined [A | B] matrix, windows of `roi_width` rows (epilogos_b200.region_null), handed to step 4 or written to
    temp_regionNull_<tag>_<file>.npz."""
    if saliency not in (1, 2):
        raise ValueError("Please ensure that saliency metric is either 1 or 2 for Pairwise Epilogos")
    if region_permutations > 0 and region_seed is None:
        raise ValueError("region permutations need the run's region seed (region_null.region_seed), drawn once per run")
    null_mode = null_mode or os.environ.get("EPILOGOS_B200_NULL", "device")
    if null_mode not in ("reference", "device"):
        raise ValueError("null_mode must be 'reference' or 'device'")
    be = session.get_backend(backend)
    shard = session.load_shard(file1Path, file2Path, numStates, backend, group=group)
    c1, c2 = shard.states_a.shape[1], shard.states_b.shape[1]
    size_a, size_b = shuffled_widths(c1, c2, groupSize)                            # helpers.py:190-194
    exp = be.to_device(np.load(expFreqPath, allow_pickle=False))

    cnt_a, cnt_b = shard.counts("a"), shard.counts("b")
    draw_seed = file_seed(run_seed(seed), filename) if null_mode == "device" or permutations > 0 else None
    if null_mode == "reference":
        rows = shard.states_a.shape[0]
        perm = np.argsort(np.random.rand(rows, c1 + c2), axis=1)                     # helpers.py:183
        null_a, null_b = be.shuffled_counts_perm(shard.states_a, shard.states_b, perm, numStates, size_a, size_b)
    else:
        null_a, null_b = be.shuffled_counts_device(cnt_a, cnt_b, size_a, size_b, draw_seed, nperm, width=c1 + c2,
                                                   bin_offset=shard.lo)

    # S1 observes over the width of the array it is given (scores.py:343); S2 normalises the shuffled halves with
    # the ORIGINAL group widths even under -g (scores.py:397-398, 418-421)
    p1, p2 = c1 * (c1 - 1), c2 * (c2 - 1)
    exact = null_mode == "reference"
    score_a = be.scores(cnt_a, c1, saliency, exp, perms=p1, exact=exact)
    score_b = be.scores(cnt_b, c2, saliency, exp, perms=p2, exact=exact)
    nshape = tuple(null_a.shape)
    flat_a, flat_b = null_a.reshape(-1, numStates), null_b.reshape(-1, numStates)
    nscore_a = be.scores(flat_a, max(size_a, 1), saliency, exp, perms=p1, exact=exact)
    nscore_b = be.scores(flat_b, max(size_b, 1), saliency, exp, perms=p2, exact=exact)
    delta, _ = be.pairwise_combine(score_a, score_b, None, None)
    _, null_dist = be.pairwise_combine(None, None, nscore_a, nscore_b)
    if len(nshape) == 3:                # [nperm][rows] flat, permutation-major: row p = the p-th shuffle of every bin
        null_dist = null_dist.reshape(nshape[0], nshape[1])
    quies = be.quiescent_mask(cnt_a, c1, cnt_b, c2, quiescentState)
    exceed = None
    if permutations > 0:
        # the real distance step 4 judges: the delta row after its "%.5f" text round trip
        real_dist, _ = be.pairwise_real_reduce(delta, text_round_trip=True)
        exceed = be.permutation_exceedances(cnt_a, cnt_b, real_dist, permutations, draw_seed, size_a, size_b, c1 + c2,
                                            shard.lo, saliency, exp, (max(size_a, 1), max(size_b, 1)), (p1, p2),
                                            exact=exact)
    region = None
    if region_permutations > 0:
        from . import region_null
        region = region_null.shard_maxima(be, "paired", shard.states_device(), lambda n: _head(shard, n), (c1, c2),
                                          numStates, roi_width, region_permutations, region_seed, saliency, exp,
                                          exact=exact)

    total = shard.total_rows
    delta = dist.gather_rows(delta, total)
    quies = dist.gather_rows(quies, total)
    if null_dist.dim() == 2:            # [nperm, rows] -> gather per permutation: rank 0 gets [nperm, all rows]
        parts = [dist.gather_rows(null_dist[p].contiguous(), total) for p in range(null_dist.shape[0])]
        null_dist = None if parts[0] is None else __import__("torch").stack(parts, dim=0)
    else:
        null_dist = dist.gather_rows(null_dist, total)
    if exceed is not None:
        exceed = dist.gather_rows(exceed, total)
    loc = _gather_locations(shard)
    if dist.rank() == 0:
        outputDirPath = Path(outputDirPath)
        if region is not None:
            from . import region_null
            region_null.check_one_chromosome(loc["chrom"], file1Path)
        writer.write_scores_text(outputDirPath / "pairwiseDelta_{}_{}.txt.gz".format(fileTag, filename),
                                 delta.cpu().numpy(), loc)
        chrName = loc["chrom"][0] if len(loc["chrom"]) else ""
        nullPath = outputDirPath / "temp_nullDistances_{}_{}.npz".format(fileTag, filename)
        if session.handover_enabled and not os.environ.get("EPILOGOS_B200_KEEP_TEMP"):
            # the paired statistics stage runs next, in this process: hand over what it reads, reduced on the device to
            # the distance and the max-difference state of every bin (roi_pairwise.readInData)
            distance, max_diff = be.pairwise_real_reduce(delta, text_round_trip=True)
            session.handover[str(nullPath)] = dict(chrName=str(chrName), distance=distance, max_diff=max_diff,
                                                   null=null_dist, quiescence=quies, chrom=loc["chrom"],
                                                   start=np.asarray(loc["start"], dtype=np.int64),
                                                   end=np.asarray(loc["end"], dtype=np.int64))
            if exceed is not None:
                session.handover[str(nullPath)].update(exceedances=exceed, permutations=int(permutations))
            if region is not None:
                region_null.stage_output(outputDirPath, fileTag, filename, chrName, region.cpu().numpy(), roi_width,
                                         region_permutations, session.handover[str(nullPath)])
            return
        helpers.savez_level(nullPath, chrName=np.array([chrName]), nullDistances=null_dist.cpu().numpy())
        helpers.savez_level(outputDirPath / "temp_quiescence_{}_{}.npz".format(fileTag, filename),
                            chrName=np.array([chrName]), quiescenceArr=quies.cpu().numpy().astype(np.bool_))
        if exceed is not None:
            helpers.savez_level(outputDirPath / "temp_permutations_{}_{}.npz".format(fileTag, filename),
                                chrName=np.array([chrName]), exceedances=exceed.cpu().numpy().view(np.uint32),
                                permutations=np.array(int(permutations), dtype=np.int64))
        if region is not None:
            region_null.stage_output(outputDirPath, fileTag, filename, chrName, region.cpu().numpy(), roi_width,
                                     region_permutations, None)


def _head(shard, n):
    """The first n rows of the shard's combined [A | B] label matrix, on the host."""
    a = shard.states_a.head(n) if hasattr(shard.states_a, "head") else np.asarray(shard.states_a[:n])
    if not shard.paired:
        return a
    b = shard.states_b.head(n) if hasattr(shard.states_b, "head") else np.asarray(shard.states_b[:n])
    return np.concatenate((a, b), axis=1)
