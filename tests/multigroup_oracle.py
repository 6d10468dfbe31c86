"""numpy definitions of the multi-group statistic, its driver and the permutation counts (include/epilogos_b200.h,
csrc/multigroup.cu).  The loops run in the specified order and every operation is one float64 numpy operation, rounded
once, so the device's numbers are reproduced bit for bit.  Each operation is vectorised over bins only."""
import numpy as np


def statistic(scores, sizes):
    """scores float32 [G, bins, K] -> (T float64 [bins], m float64 [K, bins])."""
    G, bins, K = scores.shape
    N = float(sum(sizes))
    n = [float(x) for x in sizes]
    sc = scores.astype(np.float64)
    m = np.empty((K, bins))
    t = np.zeros(bins)
    for s in range(K):
        acc = np.zeros(bins)
        for g in range(G):
            acc = acc + n[g] * sc[g, :, s]
        m[s] = acc / N
        for g in range(G):
            d = sc[g, :, s] - m[s]
            t = t + n[g] * (d * d)
    return t / N, m


def stat_and_driver(scores, sizes):
    """(T, g*, s*, sign) per bin: g* = argmax_g n_g sum_s (S_g[s] - m[s])^2, s* = argmax_s |S_g*[s] - m[s]| (first on
    ties), sign = -1 where S_g*[s*] < m[s*], else +1."""
    G, bins, K = scores.shape
    t, m = statistic(scores, sizes)
    sc = scores.astype(np.float64)
    best_v = np.full(bins, -1.0)
    best_g = np.zeros(bins, dtype=np.int64)
    for g in range(G):
        acc = np.zeros(bins)
        for s in range(K):
            d = sc[g, :, s] - m[s]
            acc = acc + d * d
        v = float(sizes[g]) * acc
        better = v > best_v
        best_v = np.where(better, v, best_v)
        best_g = np.where(better, g, best_g)
    rows = np.arange(bins)
    best_d = np.full(bins, -1.0)
    sel = np.zeros(bins)
    best_s = np.zeros(bins, dtype=np.int64)
    for s in range(K):
        d = sc[best_g, rows, s] - m[s]
        better = np.abs(d) > best_d
        best_d = np.where(better, np.abs(d), best_d)
        sel = np.where(better, d, sel)
        best_s = np.where(better, s, best_s)
    return t, best_g, best_s, np.where(sel < 0, -1, 1)


def exceedances(null_scores, sizes, t):
    """k[b] = #{p : T of null_scores[p] (float32 [P, G, bins, K]) >= t[b]}."""
    k = np.zeros(null_scores.shape[2], dtype=np.int64)
    for p in range(null_scores.shape[0]):
        k += statistic(null_scores[p], sizes)[0] >= t
    return k


def pvalues(k, nperm):
    """p = (1 + k) / (P + 1)."""
    return (1.0 + np.asarray(k, dtype=np.float64)) / (nperm + 1.0)
