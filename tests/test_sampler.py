"""The numpy restatement of the device's random streams (tests/sampler_oracle.py) checked on its own, without a device:
Philox against the Random123 known answers, the chained hypergeometric draws against the exact multivariate
hypergeometric law, the float64 inversion against exact rational inversion, and the keyed subsample's permutation.  The
device is compared with the restatement in test_sampler_gpu.py."""
import itertools
import math
from fractions import Fraction

import numpy as np
import pytest

import sampler_oracle as so


@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, want):
    assert " ".join("%08x" % int(w) for w in so.philox(ctr, key)) == want


def test_stream_word_order_and_counter():
    """Words come out as out[3], out[2], out[1], out[0] of block 0, then of block 1 (ctr[0] + 1)."""
    seed, p, gb = 0x0123456789ABCDEF, 5, (3 << 32) + 9
    st = so.shuffle_streams(seed, [p], [gb])
    got = [int(st.next(np.array([0]))[0]) for _ in range(8)]
    key = (seed & 0xFFFFFFFF, seed >> 32)
    b0 = so.philox((0, p, 9, 3), key)
    b1 = so.philox((1, p, 9, 3), key)
    assert got == [int(w) for w in (b0[3], b0[2], b0[1], b0[0], b1[3], b1[2], b1[1], b1[0])]


def test_uniform53_is_the_float64_expression():
    top = np.uint64(0xFFFFFFFF)
    assert so.uniform53(np.array([top]), np.array([top]))[0] == 1.0              # 2^53 - 1 + 0.5 rounds up to even
    assert so.uniform53(np.array([np.uint64(0)]), np.array([np.uint64(0)]))[0] == 0.5 / 2.0 ** 53
    hi, lo = np.uint64(0x80000000), np.uint64(0x40)
    # 2^52 + 1 + 0.5 is a tie at a spacing of 1: it rounds to the even 2^52 + 2
    assert so.uniform53(np.array([hi]), np.array([lo]))[0] == (2.0 ** 52 + 2.0) / 2.0 ** 53


def exact_pmf(N, K, n, x):
    if x < 0 or x > K or n - x < 0 or n - x > N - K:
        return Fraction(0)
    return Fraction(math.comb(K, x) * math.comb(N - K, n - x), math.comb(N, n))


def compositions(total, parts, caps):
    """Every vector of `parts` nonnegative integers summing to `total` with v[i] <= caps[i]."""
    if parts == 1:
        if total <= caps[0]:
            yield (total,)
        return
    for v in range(min(total, caps[0]) + 1):
        for rest in compositions(total - v, parts - 1, caps[1:]):
            yield (v,) + rest


def chain_probability(steps, forced):
    """Product over the draws of the exact pmf of the forced outcome at the draw's (N, K, n); steps without a draw have
    zero parameters and must be forced to 0."""
    prob = Fraction(1)
    for (N, K, n), x in zip(steps, forced):
        if N == 0 and K == 0 and n == 0:
            if x != 0:
                return Fraction(0)
            continue
        prob *= exact_pmf(int(N), int(K), int(n), int(x))
    return prob


def multinomial(total, parts):
    out = math.factorial(total)
    for v in parts:
        out //= math.factorial(v)
    return out


@pytest.mark.parametrize("comb, sizes", [
    ((3, 0, 2, 1), (4, 2)), ((5, 4, 3), (6, 6)), ((2, 2, 2, 2), (3, 2)), ((7, 1), (1, 1)), ((1, 1, 1, 1), (2, 2)),
    ((4, 4, 4), (5, 3)), ((0, 6, 0, 0), (3, 3)),
])
def test_paired_chain_is_the_multivariate_hypergeometric_law(comb, sizes):
    """Every (A', B') split: the chained draws of draw_shuffle, conditioned on it, give exactly
    prod_s C(c_s, a_s) C(c_s - a_s, b_s) / (C(R, n_a) C(R - n_a, n_b)); with or without -g (sizes below the row)."""
    K, R = len(comb), sum(comb)
    na = min(sizes[0], R)
    nb = min(sizes[1], R - na)
    outcomes = [(a, b) for a in compositions(na, K, comb)
                for b in compositions(nb, K, [c - x for c, x in zip(comb, a)])]
    fa = np.array([o[0] for o in outcomes])
    fb = np.array([o[1] for o in outcomes])
    M = len(outcomes)
    ca = np.tile(np.array(comb), (M, 1))
    r = so.draw_shuffle(99, np.zeros(M, dtype=np.int64), np.arange(M), ca, np.zeros_like(ca), sizes[0], sizes[1],
                        forced=(fa, fb))
    total = Fraction(0)
    for i, (a, b) in enumerate(outcomes):
        steps, xs = [], []
        for s in range(K):
            steps += [r["pa"][i, s], r["pb"][i, s]]
            xs += [a[s], b[s]]
        got = chain_probability(steps, xs)
        want = Fraction(math.prod(math.comb(c, x) * math.comb(c - x, y) for c, x, y in zip(comb, a, b)),
                        math.comb(R, na) * math.comb(R - na, nb))
        assert got == want, (a, b)
        total += got
    assert total == 1


@pytest.mark.parametrize("comb, sizes", [
    ((3, 2, 1, 2), (3, 3, 2)), ((4, 0, 5), (2, 3, 4)), ((2, 2, 2), (2, 2, 2)), ((3, 3, 1, 1), (1, 2, 3)),
    ((5, 4), (3, 3, 3)), ((1, 2, 3), (1, 1, 1)), ((6, 2), (4, 4)),
])
def test_multigroup_chain_is_the_multivariate_hypergeometric_law(comb, sizes):
    """Every assignment of the labels to G <= 3 groups (sizes covering the row or not): the chained draws of
    draw_multigroup_shuffle give exactly prod_s multinomial(c_s; x_0s, .., x_Gs, rest) / multinomial(R; n_0, .., rest)."""
    K, G, R = len(comb), len(sizes), sum(comb)
    needs, left = [], R
    for n in sizes:
        needs.append(min(n, left))
        left -= needs[-1]

    def assign(g, caps):
        if g == G:
            yield ()
            return
        for v in compositions(needs[g], K, caps):
            for rest in assign(g + 1, [c - x for c, x in zip(caps, v)]):
                yield (v,) + rest

    outcomes = list(assign(0, list(comb)))
    forced = np.array(outcomes)                                   # [M, G, K]
    M = len(outcomes)
    r = so.draw_multigroup_shuffle(7, np.zeros(M, dtype=np.int64), np.arange(M), np.tile(np.array(comb), (M, 1)),
                                   sizes, forced=forced)
    total = Fraction(0)
    for i, out in enumerate(outcomes):
        steps = [r["p"][i, g, s] for s in range(K) for g in range(G)]
        xs = [out[g][s] for s in range(K) for g in range(G)]
        got = chain_probability(steps, xs)
        num = math.prod(multinomial(comb[s], [out[g][s] for g in range(G)] + [comb[s] - sum(o[s] for o in out)])
                        for s in range(K))
        want = Fraction(num, multinomial(R, needs + [R - sum(needs)]))
        assert got == want, out
        total += got
    assert total == 1


def test_float64_inversion_equals_exact_rational_inversion():
    """Random U on random HG(N, K, n) with N <= 200: the walk-order inversion from float64 log-factorial pmfs picks the
    outcome exact rational inversion picks, except within 1e-12 of a cumulative boundary (none expected)."""
    rng = np.random.default_rng(12)
    N = rng.integers(2, 201, size=400)
    K = np.array([rng.integers(1, n) for n in N])
    n = np.array([rng.integers(1, m) for m in N])
    U = (rng.integers(0, 2 ** 53, size=len(N), dtype=np.uint64).astype(np.float64) + 0.5) / 2.0 ** 53
    U[:40] = rng.random(40) * 1e-6                         # the lower tail
    U[40:80] = 1.0 - rng.random(40) * 1e-9                 # the far upper tail
    x, margin = so.hg_invert(U, N, K, n)
    lo, hi, mode = so.hg_support(N, K, n)
    excluded = 0
    for i in range(len(N)):
        u = Fraction(float(U[i]))
        order = [int(mode[i])]
        for t in range(1, int(hi[i] - lo[i]) + 1):
            order += [v for v in (mode[i] + t, mode[i] - t) if lo[i] <= v <= hi[i]]
        cum, want = Fraction(0), None
        for v in order:
            cum += exact_pmf(int(N[i]), int(K[i]), int(n[i]), int(v))
            if u <= cum:
                want = int(v)
                break
        assert want is not None
        assert so.walk_position(want, lo[i], hi[i], mode[i]) == order.index(want)
        if margin[i] <= 1e-12:
            excluded += 1
            continue
        assert x[i] == want, (N[i], K[i], n[i], U[i])
    assert excluded == 0


@pytest.mark.parametrize("h", range(1, 9))
def test_feistel_is_a_bijection(h):
    v = np.arange(4 ** h, dtype=np.uint64)
    for seed, trial in ((0, 0), (0xDEADBEEF12345678, 7), (5, 65534)):
        img = so.feistel(v, h, seed, trial)
        assert np.array_equal(np.sort(img), v)
    assert not np.array_equal(so.feistel(v, h, 1, 0), so.feistel(v, h, 1, 1)) or h == 1


SUBSAMPLE_N = [1, 2, 3, 5, 100000, 100001, 1 << 16, (1 << 16) + 1, 1 << 17, (1 << 17) + 1, 1234567, 15500000,
               (1 << 31) - 1]


@pytest.mark.parametrize("n", SUBSAMPLE_N)
def test_cycle_walking_gives_distinct_indices(n):
    bits, h = so.subsample_bits(n)
    assert (1 << bits) >= n and (bits == 1 or (1 << (bits - 1)) < n) and h == (bits + 1) // 2
    size = min(n, 100000)
    idx = so.null_subsample(n, 2, size, 0x1234567890ABCDEF)
    assert idx.shape == (2, size) and idx.min() >= 0 and idx.max() < n
    for row in idx:
        assert len(np.unique(row)) == size
    if n == size:
        assert np.array_equal(np.sort(idx[0]), np.arange(n))
