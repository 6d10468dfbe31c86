"""Every device draw against the numpy restatement of its stream (tests/sampler_oracle.py): the paired and multi-group
shuffle samplers outcome by outcome, the fused S1 permutation counts from the restatement's draws alone, a seeded paired
run on the stand-in backend against the same run on the device, and every index of the keyed null subsample.

Comparison rule for the shuffle draws: each (permutation, bin, state[, group]) outcome equals the restatement's wherever
the restatement's margin (the distance from U to the nearest cumulative boundary next to its outcome) exceeds 1e-8.
Both sides compute pmf(mode) from log-factorials; at widths up to 12,798, log(12,799!) ~ 1.1e5, whose last-bit
differences between the device's lgamma/exp and the host's move a boundary by ~1e-9 at most.  The restatement conditions
every step on the device's earlier outcomes, so one near-tie does not cascade; draws inside the margin are counted
(expected none, at most 10 allowed) and must be the restatement's outcome or its neighbour in the walk order."""
import ctypes

import numpy as np
import pytest

import multigroup_oracle as mgo
import sampler_oracle as so
from oracle import epilogos_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

MARGIN = 1e-8
MAX_EXCLUDED = 10
SEED_HI = 0xC0FFEE1500000000            # every seed here has a nonzero high word


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import build, engine
    build.build()
    engine.device_info()
    return engine


def dev16(a):
    return torch.from_numpy(np.ascontiguousarray(a).astype(np.uint16).view(np.int16)).cuda()


def host(t):
    return t.cpu().numpy().view(np.uint16).astype(np.int64)


def check_draws(what, ref, margin, got, params):
    """got == ref wherever margin > MARGIN; inside the margin, got is ref or its neighbour in the walk order.  Prints
    the outcomes compared and those inside the margin."""
    close = margin <= MARGIN
    bad = (ref != got) & ~close
    assert not bad.any(), "%s: %d outcomes differ from the restatement, first at %s: device %d, restatement %d" % (
        what, bad.sum(), np.argwhere(bad)[0], got[bad][0], ref[bad][0])
    for i in np.argwhere(close & (ref != got)):
        N, K, n = params[tuple(i)]
        lo, hi, mode = (int(v[0]) for v in so.hg_support([N], [K], [n]))
        step = so.walk_position(got[tuple(i)], lo, hi, mode) - so.walk_position(ref[tuple(i)], lo, hi, mode)
        assert abs(step) == 1, (what, i, got[tuple(i)], ref[tuple(i)])
    excluded = int(close.sum())
    print("%s: %d outcomes compared, %d inside the %.0e margin" % (what, ref.size - excluded, excluded, MARGIN))
    assert excluded <= MAX_EXCLUDED, what


def labels_to_counts(x, K):
    return orc.bin_counts(x, K).astype(np.int64)


def crafted_rows(width, K, rng):
    """Bins of `width` labels: all one state (each end of the state range), one odd label, every state present (each
    once, the rest in the last state)."""
    rows = [np.zeros(width, dtype=np.int64), np.full(width, K - 1)]
    if K > 1:
        odd = np.zeros(width, dtype=np.int64)
        odd[rng.integers(width)] = K - 1
        rows.append(odd)
        if width >= K:
            every = np.full(width, K - 1)
            every[:K] = np.arange(K)
            rows.append(rng.permutation(every))
    return np.stack(rows)


def paired_rows(c1, c2, K, bins, kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "all":                                  # every (A, B) count vector of one label each
        a = np.repeat(np.arange(K), K)[:, None]
        b = np.tile(np.arange(K), K)[:, None]
        x = np.concatenate([a, b], axis=1)
    elif K == 1:
        x = np.zeros((bins, c1 + c2), dtype=np.int64)
    else:
        x = orc.synth_states(bins, c1 + c2, K, seed).astype(np.int64)
        if kind == "sparse":                           # many states empty or single
            x = np.where(rng.random(x.shape) < 0.97, x, rng.integers(0, K, size=x.shape))
    x = np.concatenate([x, crafted_rows(c1 + c2, K, rng)])
    return labels_to_counts(x[:, :c1], K), labels_to_counts(x[:, c1:], K)


PAIRED = [  # c1, c2, K, -g, bins, kind, perm_offset, nperm, bin_offset
    (400, 433, 18, -1, 4096, "realistic", 0, 32, 0),
    (60, 67, 15, 50, 2000, "realistic", (1 << 32) - 8, 8, (1 << 33) + 3),
    (60, 67, 15, 100, 500, "realistic", 0, 8, 7),
    (17, 16, 32, -1, 1000, "sparse", 0, 16, 0),
    (1, 1, 2, -1, 0, "all", 0, 64, 0),
    (6399, 6399, 18, -1, 64, "realistic", 0, 4, 0),      # (2 width + 3) doubles: the shared-memory limit
    (9, 9, 1, -1, 10, "realistic", 0, 4, 0),             # one state: every draw degenerate, no word consumed
]


@pytest.mark.parametrize("case", PAIRED, ids=lambda c: "%d+%d_k%d_g%d" % c[:4])
def test_paired_draws_equal_the_restatement(eng, case):
    from epilogos_b200.pairwise import shuffled_widths
    c1, c2, K, g, bins, kind, p0, P, off = case
    ca, cb = paired_rows(c1, c2, K, bins, kind, seed=c1 + c2 + K)
    rows = len(ca)
    size_a, size_b = shuffled_widths(c1, c2, g)
    seed = SEED_HI | (c1 * 1000 + c2)
    oa, ob = eng.shuffled_counts_philox_range(dev16(ca), dev16(cb), size_a, size_b, seed, p0, P, c1 + c2,
                                              bin_offset=off)
    ga, gb = host(oa).reshape(P * rows, K), host(ob).reshape(P * rows, K)
    perm = p0 + np.repeat(np.arange(P, dtype=np.int64), rows)
    gbin = off + np.tile(np.arange(rows, dtype=np.int64), P)
    r = so.draw_shuffle(seed, perm, gbin, np.tile(ca, (P, 1)), np.tile(cb, (P, 1)), size_a, size_b, forced=(ga, gb))
    check_draws("paired %s A'" % (case,), r["a"], r["ma"], ga, r["pa"])
    check_draws("paired %s B'" % (case,), r["b"], r["mb"], gb, r["pb"])
    comb = np.tile(ca + cb, (P, 1))
    assert np.all(ga + gb <= comb)
    assert np.array_equal(ga.sum(axis=1), np.minimum(size_a, comb.sum(axis=1)))
    if K == 1:
        assert np.all(r["words"] == 0)


def split(n, G):
    return [n // G + (1 if g < n % G else 0) for g in range(G)]


def multigroup_max_width(G):
    """The largest N whose sampler tables and need counts fit the kernel's 200 KB: (2 N + 3) 8 + G 256 4 <= 200 KB."""
    return ((200 * 1024 - G * 256 * 4) // 8 - 3) // 2


def test_multigroup_shared_memory_limit(eng):
    assert multigroup_max_width(2) == 12670 and multigroup_max_width(64) == 8702
    for G in (2, 64):
        n = multigroup_max_width(G) + 1
        cnt = torch.zeros((G, 1, 4), dtype=torch.int16, device="cuda")
        with pytest.raises(Exception, match="too many biosamples"):
            eng.multigroup_shuffled_counts_range(cnt, split(n, G), 1, 0, 1)


MULTI = [  # sizes, K, bins, perm_offset, nperm, bin_offset
    (split(127, 3), 15, 1000, 0, 16, 0),
    (split(833, 8), 18, 1000, (1 << 32) - 8, 8, (1 << 33) + 3),
    (split(13 * 64 + 5, 64), 25, 200, 0, 4, 7),
    ([1, 2, 500, 3], 18, 1000, 0, 8, 0),
    (split(12670, 2), 18, 48, 0, 4, (1 << 33) + 3),
    (split(8702, 64), 18, 24, (1 << 32) - 4, 4, 0),
]


@pytest.mark.parametrize("case", MULTI, ids=lambda c: "G%d_N%d_k%d" % (len(c[0]), sum(c[0]), c[1]))
def test_multigroup_draws_equal_the_restatement(eng, case):
    sizes, K, bins, p0, P, off = case
    G, N = len(sizes), sum(sizes)
    rng = np.random.default_rng(N + G)
    x = orc.synth_states(bins, N, K, N).astype(np.int64)
    x = np.concatenate([x, crafted_rows(N, K, rng)])
    rows = len(x)
    bounds = np.cumsum([0] + sizes)
    cnt = np.stack([labels_to_counts(x[:, bounds[g]:bounds[g + 1]], K) for g in range(G)])
    seed = SEED_HI | (N * 64 + G)
    out = host(eng.multigroup_shuffled_counts_range(dev16(cnt), sizes, seed, p0, P, bin_offset=off))
    got = out.reshape(P, G, rows, K).transpose(0, 2, 1, 3).reshape(P * rows, G, K)
    perm = p0 + np.repeat(np.arange(P, dtype=np.int64), rows)
    gbin = off + np.tile(np.arange(rows, dtype=np.int64), P)
    comb = np.tile(cnt.sum(axis=0), (P, 1))
    r = so.draw_multigroup_shuffle(seed, perm, gbin, comb, sizes, forced=got)
    check_draws("multigroup %s" % ((G, N, K, p0, P, off),), r["x"], r["m"], got, r["p"])
    assert np.array_equal(got.sum(axis=1), comb)                 # the sizes cover the row: every label is given out


def near_tie_bins(margins, P, rows):
    """Bins any of whose P draws has an outcome inside the margin."""
    m = margins.reshape(P, rows, -1)
    return np.flatnonzero((m <= MARGIN).any(axis=(0, 2)))


@pytest.mark.parametrize("P", [1, 7, 9, 33, 64])
@pytest.mark.parametrize("case", [(400, 433, 18, -1, 0), (60, 67, 15, 50, (1 << 33) + 1)], ids=["833", "127_g50"])
def test_fused_paired_s1_counts_from_the_restatements_draws(eng, case, P):
    """k of the fused kernel (thread groups of 1, 8 and 32, and a remainder) against the restatement's draws scored by
    the oracle (the device's S1 float32 scores are the oracle's bit for bit) and counted against the real distance."""
    from epilogos_b200.backend import CudaBackend
    from epilogos_b200.pairwise import shuffled_widths
    c1, c2, K, g, off = case
    ca, cb = paired_rows(c1, c2, K, 1500, "realistic", seed=K)
    rows = len(ca)
    size_a, size_b = shuffled_widths(c1, c2, g)
    exp = orc.normalize_expected((ca + cb).sum(axis=0))
    delta = orc.s1_scores_from_counts(ca, c1, exp) - orc.s1_scores_from_counts(cb, c2, exp)
    dist, _ = orc.paired_real_reductions(delta)
    dist = np.asarray(dist, dtype=np.float32)
    seed = SEED_HI | (P * 7 + c1)
    r = so.draw_shuffle(seed, np.repeat(np.arange(P), rows), off + np.tile(np.arange(rows), P), np.tile(ca, (P, 1)),
                        np.tile(cb, (P, 1)), size_a, size_b)
    d = orc.s1_scores_from_counts(r["a"], size_a, exp) - orc.s1_scores_from_counts(r["b"], size_b, exp)
    null = (np.sum(d * d, axis=1) * np.sign(np.sum(d, axis=1))).astype(np.float32).reshape(P, rows)
    want = (np.abs(null) >= np.abs(dist)).sum(axis=0)
    k = CudaBackend().permutation_exceedances(dev16(ca), dev16(cb), torch.from_numpy(dist).cuda(), P, seed, size_a,
                                              size_b, c1 + c2, off, 1, torch.from_numpy(exp).cuda(), (size_a, size_b),
                                              (0, 0))
    k = k.cpu().numpy().view(np.uint32).astype(np.int64)
    skip = np.union1d(near_tie_bins(r["ma"], P, rows), near_tie_bins(r["mb"], P, rows))
    keep = np.setdiff1d(np.arange(rows), skip)
    print("fused paired S1 %s P=%d: %d bins compared, %d with a draw inside the margin" % (case, P, len(keep), len(skip)))
    assert len(skip) <= MAX_EXCLUDED
    assert k[keep].tolist() == want[keep].tolist()
    assert want.max() > 0 and want.min() < P or P == 1


@pytest.mark.parametrize("P", [1, 9, 33])
@pytest.mark.parametrize("sizes", [split(127, 3), split(833, 8), [1, 2, 500, 3]], ids=["G3", "G8", "uneven"])
def test_fused_multigroup_s1_counts_from_the_restatements_draws(eng, sizes, P):
    from epilogos_b200.backend import CudaBackend
    G, N, K = len(sizes), sum(sizes), 18
    off = (1 << 33) + 1
    x = orc.synth_states(1200, N, K, N + P).astype(np.int64)
    bounds = np.cumsum([0] + sizes)
    cnt = np.stack([labels_to_counts(x[:, bounds[g]:bounds[g + 1]], K) for g in range(G)])
    rows = cnt.shape[1]
    exp = orc.normalize_expected(cnt.sum(axis=(0, 1)))
    real = np.stack([orc.s1_scores_from_counts(cnt[g], n, exp) for g, n in enumerate(sizes)])
    t, _ = mgo.statistic(real, sizes)
    seed = SEED_HI | (N * 3 + P)
    r = so.draw_multigroup_shuffle(seed, np.repeat(np.arange(P), rows), off + np.tile(np.arange(rows), P),
                                   np.tile(cnt.sum(axis=0), (P, 1)), sizes)
    xs = r["x"].reshape(P, rows, G, K)
    null = np.stack([np.stack([orc.s1_scores_from_counts(xs[p, :, g], n, exp) for g, n in enumerate(sizes)])
                     for p in range(P)]).astype(np.float32)
    want = mgo.exceedances(null, sizes, t)
    k = CudaBackend().multigroup_exceedances(dev16(cnt), sizes, torch.from_numpy(t).cuda(), P, seed, off, 1,
                                             torch.from_numpy(exp).cuda())
    k = k.cpu().numpy().view(np.uint32).astype(np.int64)
    skip = near_tie_bins(r["m"], P, rows)
    keep = np.setdiff1d(np.arange(rows), skip)
    print("fused multigroup S1 G=%d P=%d: %d bins compared, %d with a draw inside the margin" % (G, P, len(keep),
                                                                                             len(skip)))
    assert len(skip) <= MAX_EXCLUDED
    assert k[keep].tolist() == want[keep].tolist()


@pytest.mark.parametrize("group_size", [-1, 20])
def test_seeded_paired_run_on_the_stand_in_equals_the_device(eng, tmp_path, golden, monkeypatch, group_size):
    """Steps 1-3 in device null mode with one EPILOGOS_B200_SEED, S1 with 50 permutations, on the stand-in backend (the
    restatement's draws) and on CUDA: the null distances and the quiescence mask byte for byte, the counts exactly.  This
    pins the file seed, the shuffled widths and the global bin keys end to end."""
    from epilogos_b200 import expected, expectedCombination, scores, session
    from test_permutations import PermBackend
    from test_pairwise_stats import make_paired_inputs
    a, b, _ = make_paired_inputs(tmp_path, golden, chroms=("chr1",))
    fa, fb = a / "epilogos_matrix_chr1.txt.gz", b / "epilogos_matrix_chr1.txt.gz"
    monkeypatch.setenv("EPILOGOS_B200_SEED", str(SEED_HI | 77))
    monkeypatch.setenv("EPILOGOS_B200_NULL", "device")
    out = {}
    for name, be in (("cuda", None), ("stand-in", PermBackend())):
        d = tmp_path / name
        d.mkdir()
        session.clear()
        expected.main(fa, fb, 18, 1, d, "t", 1, False, backend=be)
        expectedCombination.main(d, d / "exp_freq_t.npy", "t", False, backend=be)
        scores.main(fa, fb, 18, 1, d, d / "exp_freq_t.npy", "t", 1, 17, group_size, False, backend=be, permutations=50)
        session.clear()
        out[name] = d
    for stem, key in (("temp_nullDistances", "nullDistances"), ("temp_quiescence", "quiescenceArr"),
                      ("temp_permutations", "exceedances")):
        f = "%s_t_epilogos_matrix_chr1.npz" % stem
        want, got = np.load(out["stand-in"] / f)[key], np.load(out["cuda"] / f)[key]
        assert want.dtype == got.dtype and want.tobytes() == got.tobytes(), f
    k = np.load(out["cuda"] / "temp_permutations_t_epilogos_matrix_chr1.npz")["exceedances"]
    assert k.max() > 0 and k.min() < 50


def subsample_indices_only(eng, n, trials, size, seed):
    """epi_null_subsample with indices only (no pool, no samples), which the entry point allows."""
    from epilogos_b200 import _lib
    idx = torch.empty((trials, size), dtype=torch.int32, device="cuda")
    _lib.call("epi_null_subsample", ctypes.c_void_p(0), int(n), int(trials), int(size), ctypes.c_uint64(seed),
              ctypes.c_void_p(idx.data_ptr()), ctypes.c_void_p(0), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    return idx.cpu().numpy()


S = 100000
SUBSAMPLE_N = [1, 2, 3, 5, S, S + 1, 1 << 16, (1 << 16) + 1, 1 << 17, (1 << 17) + 1, 1234567, 15500000, (1 << 31) - 1]


@pytest.mark.parametrize("n", SUBSAMPLE_N)
def test_subsample_indices_equal_the_restatement(eng, n):
    """One trial and three trials at S = min(n, 100,000) points, 101 trials at min(n, 2,000) points (the restatement
    is slow at 101 x 100,000); the samples are pool[idx] bit for bit."""
    seed = SEED_HI | n
    shapes = [(1, min(n, S)), (101, min(n, 2000)), (3, min(n, S))]
    pool = None if n >= (1 << 31) - 1 else torch.randn(n, device="cuda") * 3.0
    for trials, size in shapes:
        want = so.null_subsample(n, trials, size, seed)
        if pool is None:
            idx = subsample_indices_only(eng, n, trials, size, seed)
        else:
            i, samples = eng.null_subsample(pool, trials, size, seed)
            idx = i.cpu().numpy()
            assert samples.cpu().numpy().tobytes() == pool.cpu().numpy()[idx].tobytes()
        assert np.array_equal(idx, want), (n, trials, size)
    print("subsample n=%d: %d indices compared" % (n, sum(t * s for t, s in shapes)))


def test_subsample_at_the_grid_limit(eng):
    """65,535 trials (the grid's y limit) of 2 points from 3."""
    pool = torch.tensor([0.5, -1.5, 2.5], device="cuda")
    idx, samples = eng.null_subsample(pool, 65535, 2, SEED_HI | 3)
    idx = idx.cpu().numpy()
    assert np.array_equal(idx, so.null_subsample(3, 65535, 2, SEED_HI | 3))
    assert samples.cpu().numpy().tobytes() == pool.cpu().numpy()[idx].tobytes()
