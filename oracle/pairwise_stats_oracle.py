"""Oracle of the paired statistics stage (epilogos_b200.roi_pairwise; roiAndVisualPairwise.py:177-242, 339-354), pinned
to the libraries the reference calls: scipy.stats.gennorm for the fits and p-values, and a numpy restatement of
statsmodels' multipletests(method="fdr_bh").  The column layout of the text files is the one DESIGN.md documents."""
import numpy as np
import scipy.special
import scipy.stats

from . import roi_oracle
from .epilogos_oracle import paired_real_reductions, text_round_trip  # noqa: F401  (the "%.5f" round trip)


def null_pool(null_dists, quiescences):
    """Per-chromosome null distances (float32 [B] or [nperm, B], already in chromosome order) and quiescence masks ->
    the pool of the non-quiescent bins, permutation-major within a chromosome."""
    parts = []
    for null, q in zip(null_dists, quiescences):
        null = np.atleast_2d(np.asarray(null, dtype=np.float32))
        parts.append(null[:, ~np.asarray(q, dtype=bool)].ravel())
    return np.concatenate(parts)


def fit(points):
    """scipy.stats.gennorm.fit of float64 points -> (beta, loc, scale, NLL = _penalized_nnlf at the result)."""
    x = np.asarray(points, dtype=np.float64)
    beta, loc, scale = scipy.stats.gennorm.fit(x)
    return beta, loc, scale, float(scipy.stats.gennorm._penalized_nnlf((beta, loc, scale), x))


def fit_trials(pool, idx):
    """One fit per row of the index matrix int [T, S] into the pool: float64 [T, 4] (beta, loc, scale, NLL)."""
    pool = np.asarray(pool, dtype=np.float32)
    return np.array([fit(pool[np.asarray(row)]) for row in idx], dtype=np.float64)


def median_trial(nll):
    """Trials sorted by NLL, ties by index: the trial at position (T - 1) // 2."""
    nll = np.asarray(nll, dtype=np.float64)
    return int(np.lexsort((np.arange(len(nll)), nll))[(len(nll) - 1) // 2])


def pvalues(x, beta, loc, scale):
    """Two-sided p-values 2 min(cdf, sf) of gennorm at the float32 values x."""
    x = np.asarray(x, dtype=np.float32).astype(np.float64)
    d = scipy.stats.gennorm(beta, loc=loc, scale=scale)
    return np.minimum(1.0, 2.0 * np.minimum(d.cdf(x), d.sf(x)))


def pvalues_gammaincc(x, beta, loc, scale):
    """The same p-values as Q(1/beta, (|x - loc| / scale)^beta), free of the 1 - cdf cancellation."""
    x = np.asarray(x, dtype=np.float32).astype(np.float64)
    return scipy.special.gammaincc(1.0 / beta, (np.abs(x - loc) / scale) ** beta)


def bh(p):
    """statsmodels multipletests(p, method="fdr_bh")[1]: sort ascending, p_sorted / (rank / n) in float64, reverse
    cumulative minimum, clip at 1, back to input order."""
    p = np.asarray(p, dtype=np.float64)
    n = len(p)
    if n == 0:
        return p.copy()
    order = np.argsort(p, kind="stable")
    raw = p[order] / (np.arange(1, n + 1) / float(n))
    adj = np.minimum.accumulate(raw[::-1])[::-1]
    adj[adj > 1] = 1
    out = np.empty(n, dtype=np.float64)
    out[order] = adj
    return out


def metrics_text(chrom, starts, ends, state_names, max_diff, distance, p=None, q=None):
    """pairwiseMetrics_<tag>.txt lines: chrom, start, end, max-difference state, "{:.5f}" of |distance|, sign
    [, "{:.5e}" p, "{:.5e}" BH]."""
    lines = []
    for i in range(len(distance)):
        d = float(np.float32(distance[i]))
        line = "{}\t{}\t{}\t{}\t{:.5f}\t{}".format(chrom[i], int(starts[i]), int(ends[i]), state_names[max_diff[i] - 1],
                                                   abs(d), "+" if d >= 0 else "-")
        if p is not None:
            line += "\t{:.5e}\t{:.5e}".format(float(p[i]), float(q[i]))
        lines.append(line + "\n")
    return "".join(lines)


def roi_text(chrom, starts, ends, state_names, max_diff, distance, window, p=None, q=None):
    """regionsOfInterest_<tag>.txt of paired mode: roi_oracle.max_mean on |distance| (100 regions); state and sign from
    the first bin of the window with the largest |distance| [, its p and BH]."""
    absd = np.abs(np.asarray(distance, dtype=np.float32))
    sel = roi_oracle.max_mean(starts, ends, absd.astype(np.float64), window, 100)
    half = window // 2
    lines = []
    for i, idx in enumerate(sel["original_idx"]):
        lo, hi = idx - half, idx + half + (1 if window % 2 else 0)
        b = lo + int(np.argmax(absd[lo:hi]))
        line = "{}\t{}\t{}\t{}\t{:.5f}\t{}".format(chrom[idx], int(sel["start"][i]), int(sel["end"][i]),
                                                   state_names[max_diff[b] - 1], float(np.float32(sel["rolling_max"][i])),
                                                   "+" if distance[b] >= 0 else "-")
        if p is not None:
            line += "\t{:.5e}\t{:.5e}".format(float(p[b]), float(q[b]))
        lines.append(line + "\n")
    return "".join(lines)
