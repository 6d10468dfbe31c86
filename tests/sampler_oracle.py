"""numpy restatement of every random stream the device draws: Philox4x32-10 (csrc/common.cuh), the shuffle sampler of
csrc/paired_draw.cuh (shuffle_stream, uniform53, hypergeometric, draw_shuffle, draw_multigroup_shuffle) and the keyed
null subsample of csrc/pairwise_stats.cu (feistel, null_subsample_kernel).  It is the definition of what a seed draws: a
change to the device sampler changes this file in the same diff.  Test infrastructure only: the product never imports it.

Everything is vectorised over draws; the 32 x 32 bit multiplies run in uint64.  The hypergeometric outcome is found by
inversion in the device's walk order, but from pmfs computed independently from log-factorials in float64 (not the
walk's ratio products), and every draw also returns its margin: the distance from U to the nearest cumulative boundary
next to the outcome.  Where the margin is below the rounding of either side, the device may pick the neighbour.

The chained draws take optional `forced` outcomes: each step is then conditioned on the forced (device) outcomes of the
earlier steps, so one near-tie does not cascade through the rest of a draw."""
import numpy as np
from scipy.special import gammaln

M32 = np.uint64(0xFFFFFFFF)
MUL0, MUL1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
BUMP0, BUMP1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
FEISTEL_ROUNDS = 8
FEISTEL_TAG = 0x5EED5A3D


def _u64(x):
    return np.asarray(x, dtype=np.uint64) & M32


def philox(ctr, key):
    """Philox4x32-10: counter words (c0, c1, c2, c3) and key words (k0, k1), arrays of 32-bit values (broadcast together)
    -> the four output words as uint64 arrays.  Per round, with hi/lo the halves of the 64-bit products
    0xD2511F53 * c0 and 0xCD9E8D57 * c2: (hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0); the key is bumped after each round."""
    c = np.broadcast_arrays(*[_u64(w) for w in ctr])
    c = [w.copy() for w in c]
    k0, k1 = _u64(key[0]), _u64(key[1])
    for _ in range(10):
        p0, p1 = c[0] * MUL0, c[2] * MUL1
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0, k1 = (k0 + BUMP0) & M32, (k1 + BUMP1) & M32
    return c


class Streams:
    """Many Philox streams at once (Philox::next): a refill encrypts the counter and then increments ctr[0]; the words of
    a block are handed out as out[3], out[2], out[1], out[0]."""

    def __init__(self, key, ctr):
        parts = np.broadcast_arrays(*[_u64(w) for w in (*key, *ctr)])
        self.key = [w.copy() for w in parts[:2]]
        self.ctr = [w.copy() for w in parts[2:]]
        self.out = np.zeros((4,) + self.ctr[0].shape, dtype=np.uint64)
        self.have = np.zeros(self.ctr[0].shape, dtype=np.int64)
        self.words = np.zeros(self.ctr[0].shape, dtype=np.int64)       # words consumed per stream

    def next(self, sel):
        """The next word of the streams `sel` (an index array)."""
        empty = sel[self.have[sel] == 0]
        if len(empty):
            out = philox([c[empty] for c in self.ctr], [k[empty] for k in self.key])
            for i in range(4):
                self.out[i, empty] = out[i]
            self.ctr[0][empty] = (self.ctr[0][empty] + np.uint64(1)) & M32
            self.have[empty] = 4
        h = self.have[sel] - 1
        self.have[sel] = h
        self.words[sel] += 1
        return self.out[h, sel]


def shuffle_streams(seed, perm, gbin):
    """shuffle_stream: key = (seed low word, seed high word), ctr = (0, permutation, global bin low, global bin high)."""
    seed = int(seed) & (2 ** 64 - 1)
    gbin = np.asarray(gbin, dtype=np.uint64)
    return Streams((seed & 0xFFFFFFFF, seed >> 32), (0, perm, gbin & M32, gbin >> np.uint64(32)))


def uniform53(hi, lo):
    """((hi >> 5) * 2^26 + (lo >> 6) + 0.5) * 2^-53 in float64 as written: not the exact rational, because the + 0.5
    rounds to even once the integer part reaches 2^52 (then U = 1.0 is possible, with probability 2^-53)."""
    return ((hi >> np.uint64(5)).astype(np.float64) * 67108864.0 + (lo >> np.uint64(6)).astype(np.float64) + 0.5) * \
        (1.0 / 9007199254740992.0)


_LF = np.zeros(1)


def log_factorials(n):
    """log(i!) for i = 0..n (at least), float64."""
    global _LF
    if len(_LF) <= n:
        _LF = gammaln(np.arange(max(n + 1, 2 * len(_LF)), dtype=np.float64) + 1.0)
    return _LF


def hg_pmf(N, K, n, x):
    """P(X = x) of HG(population N, K successes, n draws) from log-factorials."""
    lf = log_factorials(int(np.max(N)) if np.size(N) else 0)
    return np.exp((lf[K] - lf[x] - lf[K - x]) + (lf[N - K] - lf[n - x] - lf[N - K - n + x]) - (lf[N] - lf[n] - lf[N - n]))


def hg_support(N, K, n):
    """(lo, hi, mode) of HG(N, K, n): mode = floor((n + 1)(K + 1) / (N + 2)) clamped to [lo, hi]."""
    N, K, n = (np.asarray(v, dtype=np.int64) for v in (N, K, n))
    lo, hi = np.maximum(0, n - (N - K)), np.minimum(n, K)
    return lo, hi, np.clip(((n + 1) * (K + 1)) // (N + 2), lo, hi)


def walk_position(x, lo, hi, mode):
    """Position of outcome x in the walk order mode, mode+1, mode-1, mode+2, ... (an exhausted side skipped)."""
    t = abs(int(x) - int(mode))
    if t == 0:
        return 0
    if x > mode:                                   # after the mode, t - 1 values above and up to t - 1 below
        return t + min(t - 1, int(mode) - int(lo))
    return t + min(t, int(hi) - int(mode))         # after the mode, up to t values above and t - 1 below


def hg_invert(U, N, K, n):
    """Outcome and margin of the walk-order inversion of U for HG(N, K, n) (arrays, lo < hi everywhere): the first value
    in the order mode, mode+1, mode-1, mode+2, ... whose cumulative pmf reaches U; if none does (U above the rounded total
    mass), the residual rule of hypergeometric(): the heavier end of the support, the upper one on a tie."""
    U = np.asarray(U, dtype=np.float64)
    N, K, n = (np.asarray(v, dtype=np.int64) for v in (N, K, n))
    lo, hi, mode = hg_support(N, K, n)
    x = np.full(U.shape, -1, dtype=np.int64)
    margin = np.zeros(U.shape)
    cum = hg_pmf(N, K, n, mode)
    done = U <= cum
    x[done], margin[done] = mode[done], np.minimum(U - 0.0, cum - U)[done]
    live = np.flatnonzero(~done)
    t = 0
    while len(live):
        t += 1
        for sign in (1, -1):
            v = mode[live] + sign * t
            ok = (v <= hi[live]) & (v >= lo[live])
            i, v = live[ok], v[ok]
            before = cum[i]
            after = before + hg_pmf(N[i], K[i], n[i], v)
            cum[i] = after
            hit = U[i] <= after
            x[i[hit]] = v[hit]
            margin[i[hit]] = np.minimum(U[i] - before, after - U[i])[hit]
            live = live[x[live] < 0]
        out = (mode[live] + t >= hi[live]) & (mode[live] - t <= lo[live])
        i = live[out]
        if len(i):                                            # walked out: the rounding residue
            heavy = hg_pmf(N[i], K[i], n[i], hi[i]) >= hg_pmf(N[i], K[i], n[i], lo[i])
            x[i] = np.where(heavy, hi[i], lo[i])
            margin[i] = U[i] - cum[i]
            live = live[~out]
    return x, margin


def hypergeometric(streams, sel, N, K, n):
    """hypergeometric() for the streams `sel`: (x, margin).  lo >= hi returns lo and consumes no word (margin inf);
    otherwise two words make U and the walk-order inversion picks x."""
    lo, hi, _ = hg_support(N, K, n)
    x, margin = lo.copy(), np.full(lo.shape, np.inf)
    j = np.flatnonzero(lo < hi)
    if len(j):
        a = sel[j]
        w_hi = streams.next(a)
        w_lo = streams.next(a)
        x[j], margin[j] = hg_invert(uniform53(w_hi, w_lo), np.asarray(N)[j], np.asarray(K)[j], np.asarray(n)[j])
    return x, margin


def _take(forced, x, lo_hi):
    """The outcome the next steps are conditioned on: the forced one (clipped to the support) or the reference's."""
    if forced is None:
        return x
    lo, hi = lo_hi
    return np.clip(forced, lo, hi)


def draw_shuffle(seed, perm, gbin, ca, cb, size_a, size_b, forced=None):
    """draw_shuffle for draws (perm[i], gbin[i]) of rows ca[i], cb[i] ([M, K] counts): a'_s ~ HG(remaining, c_s,
    needed by A'), b'_s ~ HG(remaining - needed by A', c_s - a'_s, needed by B'); a state with c_s = 0 consumes no word.
    Returns dict(a, b [M, K] outcomes, ma, mb [M, K] margins (inf: no draw), pa, pb [M, K, 3] the (N, K, n) of each draw
    (zeros where c_s = 0), words [M] consumed).  forced = (fa, fb) conditions every step on the given earlier outcomes."""
    ca, cb = np.asarray(ca, dtype=np.int64), np.asarray(cb, dtype=np.int64)
    M, K = ca.shape
    st = shuffle_streams(seed, perm, gbin)
    comb = ca + cb
    remaining = comb.sum(axis=1)
    need_a = np.minimum(size_a, remaining)
    need_b = np.minimum(size_b, remaining - need_a)
    res = {k: np.zeros((M, K), dtype=np.int64) for k in ("a", "b")}
    res.update(ma=np.full((M, K), np.inf), mb=np.full((M, K), np.inf), pa=np.zeros((M, K, 3), dtype=np.int64),
               pb=np.zeros((M, K, 3), dtype=np.int64))
    for s in range(K):
        c = comb[:, s]
        i = np.flatnonzero(c > 0)
        pa = (remaining[i], c[i], need_a[i])
        ga, res["ma"][i, s] = hypergeometric(st, i, *pa)
        res["a"][i, s], res["pa"][i, s] = ga, np.stack(pa, axis=1)
        ga = _take(None if forced is None else forced[0][i, s], ga, hg_support(*pa)[:2])
        pb = (remaining[i] - need_a[i], c[i] - ga, need_b[i])
        gb, res["mb"][i, s] = hypergeometric(st, i, *pb)
        res["b"][i, s], res["pb"][i, s] = gb, np.stack(pb, axis=1)
        gb = _take(None if forced is None else forced[1][i, s], gb, hg_support(*pb)[:2])
        remaining = remaining - c
        need_a[i] -= ga
        need_b[i] -= gb
    res["words"] = st.words
    return res


def draw_multigroup_shuffle(seed, perm, gbin, comb, sizes, forced=None):
    """draw_multigroup_shuffle for draws (perm[i], gbin[i]) of the union's counts comb[i] ([M, K]) over the groups of
    `sizes`: for every state in order and every group in order, x_gs ~ HG(labels not yet given to groups 0..g-1, labels
    of state s not yet given, labels group g still needs); a group meeting no label of the state left consumes no word.
    Returns dict(x [M, G, K] outcomes, m [M, G, K] margins, p [M, G, K, 3] parameters, words [M]).  forced [M, G, K]
    conditions every step on the given earlier outcomes."""
    comb = np.asarray(comb, dtype=np.int64)
    M, K = comb.shape
    G = len(sizes)
    st = shuffle_streams(seed, perm, gbin)
    remaining = comb.sum(axis=1)
    left = remaining.copy()
    need = np.zeros((G, M), dtype=np.int64)
    for g in range(G):
        need[g] = np.minimum(sizes[g], left)
        left -= need[g]
    x = np.zeros((M, G, K), dtype=np.int64)
    m = np.full((M, G, K), np.inf)
    p = np.zeros((M, G, K, 3), dtype=np.int64)
    for s in range(K):
        pop, succ = remaining.copy(), comb[:, s].copy()
        for g in range(G):
            i = np.flatnonzero(succ > 0)
            prm = (pop[i], succ[i], need[g, i])
            xi, m[i, g, s] = hypergeometric(st, i, *prm)
            x[i, g, s], p[i, g, s] = xi, np.stack(prm, axis=1)
            xi = _take(None if forced is None else forced[i, g, s], xi, hg_support(*prm)[:2])
            pop -= need[g]
            succ[i] -= xi
            need[g, i] -= xi
        remaining -= comb[:, s]
    return dict(x=x, m=m, p=p, words=st.words)


def feistel(v, h, seed, trial):
    """feistel(): the keyed permutation of [0, 4^h): (L, R) = (v >> h, v & (2^h - 1)); 8 rounds of (L, R) <- (R, L ^ F)
    with F = out[0] & (2^h - 1) of Philox at ctr (R, round, trial, 0x5EED5A3D), key = the seed's two words."""
    seed = int(seed) & (2 ** 64 - 1)
    mask = np.uint64((1 << h) - 1)
    v = np.asarray(v, dtype=np.uint64)
    L, R = v >> np.uint64(h), v & mask
    key = (seed & 0xFFFFFFFF, seed >> 32)
    for r in range(FEISTEL_ROUNDS):
        F = philox((R, r, trial, FEISTEL_TAG), key)[0] & mask
        L, R = R, L ^ F
    return (L << np.uint64(h)) | R


def subsample_bits(n):
    """(bits, h): the smallest bits >= 1 with 2^bits >= n, and h = ceil(bits / 2)."""
    bits = 1
    while (1 << bits) < n:
        bits += 1
    return bits, (bits + 1) // 2


def null_subsample(n, trials, size, seed):
    """Indices int32 [trials, size] of epi_null_subsample: trial t's index i is the first image of i under the trial's
    Feistel permutation (applied at least once) that falls in [0, n)."""
    _, h = subsample_bits(n)
    v = np.tile(np.arange(size, dtype=np.uint64), trials)
    t = np.repeat(np.arange(trials, dtype=np.uint64), size)
    live = np.arange(len(v))
    while len(live):
        v[live] = feistel(v[live], h, seed, t[live])
        live = live[v[live] >= np.uint64(n)]
    return v.astype(np.int64).reshape(trials, size).astype(np.int32)
