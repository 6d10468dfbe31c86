"""Genome-wide family-wise p-values of the regions of interest (`--roi-permutations P`): a single-step max-T test over P
permutations of the biosample labels.

Statistic per bin: x_b = |distance_b| (paired mode and --compare: the float32 of epi_pairwise_real_reduce after the "%.5f"
text round trip, what step 4 ranks regions by) or T_b (--multigroup, float64).  Quantised as q(x) = rint(x * 2^24) in
int64 (round half to even; valid input is finite with 0 <= x < 2^24), so window sums are exact integers whatever the
chunking, the sharding or the number of GPUs.

Splits: permutation p of the N columns of the compared matrix ([A | B], or the groups of a multi-group comparison one
after the other in the order they were named) is rng.permutation(N) for p = 0 .. P - 1 in order, rng =
numpy.random.Generator(numpy.random.Philox(key=region_seed)); its consecutive slices of the group sizes are the groups.
One seed per run (region_seed below), so every file, rank and sharding mode uses the same P splits.  Permuted groups are
scored exactly like the real ones, so the identity split reproduces x_b bit for bit.

M_p = the largest sum of q(x) over W = --roi-width consecutive rows of one input file under split p, over all files.  A
region r (the rows step 4 already uses for it) has S_r = sum q(x_b), k_r = #{p : M_p >= S_r} and p_r = (1 + k_r)/(P + 1).
"""
import numpy as np

from . import dist

REGION_SEED_SALT = "epilogos_b200 region permutations"
MAX_PERMUTATIONS = 100000
MAX_WINDOW = 16384
SCALE = float(2 ** 24)


def region_seed(run_seed):
    """The key of the run's split generator: the run seed mixed with a constant (unrelated to the per-file null draws)."""
    from .pairwise import file_seed
    return file_seed(run_seed, REGION_SEED_SALT)


def quantise(x):
    """q(x) = rint(x * 2^24) as int64; raises ValueError for values that are not finite in [0, 2^24)."""
    x = np.asarray(x, dtype=np.float64)
    bad = ~((x >= 0.0) & (x < SCALE))
    if bad.any():
        i = int(np.flatnonzero(bad.ravel())[0])
        raise ValueError("region statistic {} at index {} is not a finite value in [0, 2^24)".format(x.ravel()[i], i))
    return np.rint(np.ldexp(x, 24)).astype(np.int64)


def split_blocks(seed, sizes, nperm, block):
    """(p0, members): the splits p0 .. p0 + n - 1 in blocks of at most `block`, drawn in order; members uint64
    [n, G - 1, ceil(N / 64)] holds the column bitsets of the first G - 1 groups (the last group is the rest)."""
    rng = np.random.Generator(np.random.Philox(key=int(seed)))
    N, G = int(sum(sizes)), len(sizes)
    words = (N + 63) // 64
    edges = np.cumsum([0] + [int(n) for n in sizes])
    for p0 in range(0, nperm, block):
        n = min(block, nperm - p0)
        members = np.zeros((n, G - 1, words * 64), dtype=np.uint8)
        for i in range(n):
            perm = rng.permutation(N)
            for g in range(G - 1):
                members[i, g, perm[edges[g]:edges[g + 1]]] = 1
        yield p0, np.packbits(members, axis=2, bitorder="little").view(np.uint64)


def shard_maxima(be, kind, x_dev, head, sizes, num_states, window, nperm, seed, saliency, exp, exact=False):
    """int64 [P] maxima of this file on every rank.  x_dev: the shard's rows of the compared matrix on the device; head(n):
    its first n rows on the host.  In rows mode the windows that start in a rank's rows may end in the rows of the ranks
    after it: each rank gets up to W - 1 such rows (dist.halo_rows), evaluates the windows starting in its own rows, and
    the ranks take the maximum."""
    halo = dist.halo_rows(head(window - 1), window - 1)
    fn = be.region_maxima_paired if kind == "paired" else be.region_maxima_multigroup
    m = fn(x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, exact=exact)
    return dist.all_reduce_max(m)


def check_one_chromosome(chrom, path):
    """The region null keys a file's maxima by its chromosome: one chromosome per input file."""
    names = np.unique(np.asarray(chrom, dtype=object).astype(str))
    if len(names) > 1:
        raise ValueError("--roi-permutations needs one chromosome per input file; {} holds {}".format(
            path, ", ".join(names[:4])))


def combine(chunks, what):
    """(maxima int64 [P], window, P) over the files of `chunks` (dicts with region_maxima, region_window,
    region_permutations), or None when no file has any.  Files that disagree on P or W raise ValueError."""
    keys = {(c.get("region_permutations"), c.get("region_window")) for c in chunks}
    if keys == {(None, None)}:
        return None
    if (None, None) in keys or len(keys) != 1:
        raise ValueError("{} on the number of region permutations or the window ({})".format(
            what, sorted(str(k) for k in keys)))
    P, W = keys.pop()
    return np.max(np.stack([np.asarray(c["region_maxima"], dtype=np.int64) for c in chunks]), axis=0), int(W), int(P)


def region_lines(chrom, starts, ends, x, window, maxima):
    """regionPermutation text: per region of regionsOfInterest (the same max-mean selection, in the same order) chrom,
    start, end, "%.5e" window mean of x, k, "%.5e" p."""
    from .roi import max_mean
    sel = max_mean(starts, ends, np.asarray(x, dtype=np.float64), window, 100)
    q = quantise(x)
    P = len(maxima)
    half = window // 2
    lines = []
    for i, idx in enumerate(sel["original_idx"]):
        lo, hi = max(idx - half, 0), idx + half + (1 if window % 2 else 0)
        s = int(q[lo:hi].sum())
        k = int(np.count_nonzero(maxima >= s))
        lines.append("%s\t%d\t%d\t%.5e\t%d\t%.5e\n" % (chrom[idx], sel["start"][i], sel["end"][i],
                                                       s / (window * SCALE), k, (1.0 + k) / (P + 1.0)))
    return "".join(lines)


def write_outputs(outputDirPath, fileTag, chrom, starts, ends, x, combined):
    """regionPermutation_<tag>.txt and regionNullMaxima_<tag>.npz {maxima, window, permutations}."""
    maxima, window, P = combined
    (outputDirPath / "regionPermutation_{}.txt".format(fileTag)).write_text(
        region_lines(chrom, starts, ends, x, window, maxima))
    np.savez(outputDirPath / "regionNullMaxima_{}.npz".format(fileTag), maxima=maxima.astype(np.int64),
             window=np.array(window, dtype=np.int64), permutations=np.array(P, dtype=np.int64))


def stage_output(outputDirPath, fileTag, filename, chrName, maxima, window, nperm, handover):
    """Step 3's result of one file: into `handover` (a dict step 4 of this process reads) or written as
    temp_regionNull_<tag>_<file>.npz {chrName, maxima, window, permutations}."""
    from . import helpers
    out = dict(region_maxima=np.asarray(maxima, dtype=np.int64), region_window=int(window),
               region_permutations=int(nperm))
    if handover is not None:
        handover.update(out)
        return
    helpers.savez_level(outputDirPath / "temp_regionNull_{}_{}.npz".format(fileTag, filename),
                        chrName=np.array([chrName]), maxima=out["region_maxima"],
                        window=np.array(window, dtype=np.int64), permutations=np.array(nperm, dtype=np.int64))


def read_temps(outputDirPath, fileTag, chunks):
    """Add the maxima of temp_regionNull_<tag>_<file>.npz to the step-4 chunks of their chromosomes (chunks handed over
    in memory already carry theirs)."""
    by_name = {c["chrName"]: c for c in chunks}
    for f in sorted(outputDirPath.glob("temp_regionNull_{}_*.npz".format(fileTag))):
        z = np.load(f, allow_pickle=False)
        c = by_name.get(str(z["chrName"][0]))
        if c is not None and "region_maxima" not in c:
            c.update(region_maxima=np.asarray(z["maxima"], dtype=np.int64), region_window=int(z["window"]),
                     region_permutations=int(z["permutations"]))
