"""numpy restatement of the stratified shuffles (csrc/strata.cu, draw_stratified_shuffle in csrc/paired_draw.cuh) and of
the stratified region splits (epilogos_b200/region_null.split_blocks with strata), built on sampler_oracle.  Test
infrastructure only: the product never imports it.

A stratified draw of (seed, permutation, global bin) runs the multi-group draw of sampler_oracle on each stratum in order,
on ONE stream: stratum h + 1 continues where stratum h left the stream.  The device returns only the sums over the
strata, so its outcomes cannot condition the steps here; instead every draw reports its smallest margin, and a caller
compares only the draws whose every step is outside its margin."""
import numpy as np

import sampler_oracle as so
from oracle import epilogos_oracle as orc


def _multigroup_on(st, comb, sizes):
    """sampler_oracle.draw_multigroup_shuffle on the streams `st` as they stand: (x [M, G, K], smallest margin [M])."""
    M, K = comb.shape
    G = len(sizes)
    remaining = comb.sum(axis=1)
    left = remaining.copy()
    need = np.zeros((G, M), dtype=np.int64)
    for g in range(G):
        need[g] = np.minimum(int(sizes[g]), left)
        left -= need[g]
    x = np.zeros((M, G, K), dtype=np.int64)
    margin = np.full(M, np.inf)
    for s in range(K):
        pop, succ = remaining.copy(), comb[:, s].copy()
        for g in range(G):
            i = np.flatnonzero(succ > 0)
            xi, m = so.hypergeometric(st, i, pop[i], succ[i], need[g, i])
            x[i, g, s] = xi
            margin[i] = np.minimum(margin[i], m)
            pop -= need[g]
            succ[i] -= xi
            need[g, i] -= xi
        remaining -= comb[:, s]
    return x, margin


def draw_stratified_shuffle(seed, perm, gbin, comb, sizes):
    """Draws (perm[i], gbin[i]) of the per-stratum counts comb [H, M, K] over the groups of sizes [H][G].  Returns
    dict(x [M, G, K] the groups' counts summed over the strata, xh [H, M, G, K] per stratum, margin [M] the smallest
    margin of any step of the draw, words [M])."""
    comb = np.asarray(comb, dtype=np.int64)
    H, M, K = comb.shape
    st = so.shuffle_streams(seed, perm, gbin)
    xh = np.zeros((H, M, len(sizes[0]), K), dtype=np.int64)
    margin = np.full(M, np.inf)
    for h in range(H):
        xh[h], m = _multigroup_on(st, comb[h], sizes[h])
        margin = np.minimum(margin, m)
    return dict(x=xh.sum(axis=0), xh=xh, margin=margin, words=st.words)


def shuffled_counts(cnt_h, sizes, seed, nperm, bin_offset=0, perm_offset=0):
    """[nperm, G, rows, K] of the stratified sampler: permutation p of row r from the stream (seed, perm_offset + p,
    GLOBAL bin bin_offset + r); cnt_h [H, rows, K]."""
    cnt_h = np.asarray(cnt_h, dtype=np.int64)
    H, rows, K = cnt_h.shape
    r = draw_stratified_shuffle(seed, perm_offset + np.repeat(np.arange(nperm), rows),
                                bin_offset + np.tile(np.arange(rows), nperm), np.tile(cnt_h, (1, nperm, 1)), sizes)
    return r["x"].reshape(nperm, rows, -1, K).transpose(0, 2, 1, 3)


def stratum_counts(x, columns, K):
    """[H, rows, K] counts of each stratum's column list (a column listed twice counted twice)."""
    return np.stack([orc.bin_counts(x[:, np.asarray(c)], K).astype(np.int64) for c in columns])


def splits(seed, positions, sizes, nperm):
    """Split p = 0 .. nperm - 1: per group, the positions it gets.  For every stratum h in order, its ascending positions
    permuted by rng.permutation(N_h); the first n[h][0] go to group 0, the next n[h][1] to group 1, ..."""
    rng = np.random.Generator(np.random.Philox(key=int(seed)))
    G = len(sizes[0])
    for _ in range(nperm):
        parts = [[] for _ in range(G)]
        for pos, n in zip(positions, sizes):
            moved = np.asarray(pos)[rng.permutation(len(pos))]
            cuts = np.cumsum([0] + list(n))
            for g in range(G):
                parts[g].append(moved[cuts[g]:cuts[g + 1]])
        yield [np.concatenate(p) for p in parts]


def file_maxima(x, K, positions, sizes, window, nperm, seed, stat):
    """int64 [nperm]: M_p of one file (compared matrix x [rows, N]) under the stratified splits of `seed`."""
    import region_oracle as ro
    out = []
    for parts in splits(seed, positions, sizes, nperm):
        cnt = np.stack([orc.bin_counts(x[:, p], K).astype(np.int64) for p in parts])
        out.append(ro.window_max(ro.q(stat(cnt)), window))
    return np.array(out, dtype=np.int64)
