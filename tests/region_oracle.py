"""numpy definitions of the region null (epilogos_b200/region_null.py, csrc/label_permutations.cu), written without the
package: the splits, their counts, the statistic of a split, the quantised window maxima and the region p-values."""
import numpy as np

from oracle import epilogos_oracle as orc
import multigroup_oracle as mgo

SEED_SALT = "epilogos_b200 region permutations"


def splits(seed, n_cols, nperm):
    """Permutation p of the columns, p = 0 .. nperm - 1, from one Philox-keyed generator."""
    rng = np.random.Generator(np.random.Philox(key=int(seed)))
    for _ in range(nperm):
        yield rng.permutation(n_cols)


def group_counts(x, K, perm, sizes):
    """[G, rows, K] counts of the groups of a split: consecutive slices of `perm` of the group sizes."""
    edges = np.cumsum([0] + list(sizes))
    return np.stack([orc.bin_counts(x[:, perm[edges[g]:edges[g + 1]]], K).astype(np.int64) for g in range(len(sizes))])


def score_fn(saliency, exp):
    if saliency == 1:
        return lambda c, n: orc.s1_scores_from_counts(c, n, exp)
    return lambda c, n: orc.s2_scores_from_counts(c, n * (n - 1), exp)


def paired_stat(cnt, sizes, saliency, exp):
    """|distance| (float32) of the two groups' counts: the text round trip of the delta rows, as step 4 reduces them."""
    score = score_fn(saliency, exp)
    delta = (np.asarray(score(cnt[0], sizes[0]), dtype=np.float32) - np.asarray(score(cnt[1], sizes[1]), dtype=np.float32))
    dist, _ = orc.paired_real_reductions(delta, round_trip=True)
    return np.abs(np.asarray(dist, dtype=np.float32))


def multigroup_stat(cnt, sizes, saliency, exp):
    score = score_fn(saliency, exp)
    sc = np.stack([score(cnt[g], n) for g, n in enumerate(sizes)]).astype(np.float32)
    return mgo.statistic(sc, sizes)[0]


def q(x):
    x = np.asarray(x, dtype=np.float64)
    assert np.all(np.isfinite(x)) and np.all(x >= 0) and np.all(x < 2.0 ** 24)
    return np.rint(np.ldexp(x, 24)).astype(np.int64)


def window_max(values, window):
    """Largest sum of `window` consecutive values, or -1 when there is no window."""
    if len(values) < window:
        return -1
    c = np.concatenate(([0], np.cumsum(values)))
    return int((c[window:] - c[:-window]).max())


def file_maxima(x, K, sizes, window, nperm, seed, stat):
    """int64 [nperm]: M_p of one file (label matrix x [rows, N], groups consecutive) under the splits of `seed`."""
    return np.array([window_max(q(stat(group_counts(x, K, perm, sizes))), window)
                     for perm in splits(seed, x.shape[1], nperm)], dtype=np.int64)


def region_text(chrom, starts, ends, x, window, maxima):
    """regionPermutation text for the max-mean regions of x."""
    from epilogos_b200.roi import max_mean
    sel = max_mean(starts, ends, np.asarray(x, dtype=np.float64), window, 100)
    qx = q(x)
    P = len(maxima)
    out = ""
    for i, idx in enumerate(sel["original_idx"]):
        lo, hi = max(idx - window // 2, 0), idx + window // 2 + window % 2
        s = int(qx[lo:hi].sum())
        k = int((maxima >= s).sum())
        out += "%s\t%d\t%d\t%.5e\t%d\t%.5e\n" % (chrom[idx], sel["start"][i], sel["end"][i], s / (window * 2.0 ** 24), k,
                                                (1.0 + k) / (P + 1.0))
    return out
