"""Permutation kernels (csrc/permutations.cu) against the composed entry points, and --null-permutations end to end on the
CUDA backend."""
import gzip

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import build, engine
    build.build()
    engine.device_info()
    return engine


def make_case(eng, bins, c1, c2, K, saliency, seed, planted=0):
    """Group counts with structure (a share of bins differs between the groups), the run's expected table, and the real
    distance of every bin as step 4 sees it."""
    rng = np.random.default_rng(seed)
    probs = rng.dirichlet(np.ones(K) * 0.3, size=4)
    kind = rng.integers(0, 4, size=bins)
    shift = rng.random(bins) < 0.3
    xa = np.stack([rng.choice(K, size=c1, p=probs[k]) for k in kind]).astype(np.int8)
    xb = np.stack([rng.choice(K, size=c2, p=probs[(k + s) % 4]) for k, s in zip(kind, shift)]).astype(np.int8)
    if planted:
        xa[:planted] = 0
        xb[:planted] = 1
    ca = eng.bin_counts(eng.pack_states(xa).cuda(), c1, K)
    cb = eng.bin_counts(eng.pack_states(xb).cuda(), c2, K)
    n1, n2 = eng.expected_tables((ca + cb).contiguous(), c1 + c2, want_s1=saliency == 1, want_s2=saliency == 2)
    exp = eng.normalize(n1 if saliency == 1 else n2)
    return ca, cb, exp


def score(eng, cnt, width, saliency, exp, perms):
    return eng.scores_s1(cnt, width, exp) if saliency == 1 else eng.scores_s2(cnt, width, exp, perms=perms)


def real_distance(eng, ca, cb, c1, c2, saliency, exp):
    sa = score(eng, ca, c1, saliency, exp, c1 * (c1 - 1))
    sb = score(eng, cb, c2, saliency, exp, c2 * (c2 - 1))
    delta, _ = eng.pairwise_combine(sa, sb, None, None)
    dist, _ = eng.pairwise_real_reduce(delta, True)
    return dist


def composed_k(eng, ca, cb, size_a, size_b, width, seed, bin_offset, nperm, saliency, exp, c1, c2, dist):
    """k from epi_shuffled_counts_philox_range + epi_scores_s1/s2 + epi_pairwise_combine, counted in numpy."""
    K = ca.shape[1]
    oa, ob = eng.shuffled_counts_philox_range(ca, cb, size_a, size_b, seed, 0, nperm, width, bin_offset=bin_offset)
    sa = score(eng, oa.reshape(-1, K), max(size_a, 1), saliency, exp, c1 * (c1 - 1))
    sb = score(eng, ob.reshape(-1, K), max(size_b, 1), saliency, exp, c2 * (c2 - 1))
    _, null = eng.pairwise_combine(None, None, sa, sb)
    null = null.reshape(nperm, -1).cpu().numpy()
    return (np.abs(null) >= np.abs(dist.cpu().numpy())).sum(axis=0).astype(np.uint32)


def sizes(c1, c2, g):
    from epilogos_b200.pairwise import shuffled_widths
    return shuffled_widths(c1, c2, g)


CASES = [  # bins, c1, c2, K, -g, nperm, bin_offset
    (1001, 400, 433, 18, -1, 64, 0),
    (777, 60, 67, 15, -1, 7, 12345),
    (513, 400, 433, 18, 300, 1, 5),
    (999, 60, 67, 15, 50, 64, 3),
    (301, 60, 67, 18, 100, 7, (1 << 33) + 1),
    (513, 700, 800, 18, -1, 33, 0),          # S1 value tables in global memory; 32-thread groups and one more permutation
    (300, 4100, 4200, 15, -1, 7, 0),         # wider than the S1 value table: S1 takes the composed route too
]


@pytest.mark.parametrize("saliency", [1, 2])
@pytest.mark.parametrize("case", CASES)
def test_backend_counts_equal_the_composed_entry_points(eng, case, saliency):
    """S1: the fused kernel; S2: the batched draw + tensor-core score + count loop, under two workspace caps."""
    from epilogos_b200.backend import CudaBackend
    bins, c1, c2, K, g, nperm, off = case
    ca, cb, exp = make_case(eng, bins, c1, c2, K, saliency, seed=bins + K)
    dist = real_distance(eng, ca, cb, c1, c2, saliency, exp)
    size_a, size_b = sizes(c1, c2, g)
    seed = 0x9E3779B97F4A7C15 ^ bins
    want = composed_k(eng, ca, cb, size_a, size_b, c1 + c2, seed, off, nperm, saliency, exp, c1, c2, dist)
    be = CudaBackend()
    args = (ca, cb, dist, nperm, seed, size_a, size_b, c1 + c2, off, saliency, exp, (max(size_a, 1), max(size_b, 1)),
            (c1 * (c1 - 1), c2 * (c2 - 1)))
    for cap in (1 << 30, 12 * K * 100):
        got = be.permutation_exceedances(*args, workspace_bytes=cap).cpu().numpy().view(np.uint32)
        assert got.tolist() == want.tolist(), (case, saliency, cap)
    assert want.max() <= nperm and (want.sum() > 0 or nperm == 1)


def test_fused_kernel_splits_and_batches(eng):
    """k does not depend on how the bins are split (global bin keys) or the permutations batched (perm_offset); the range
    sampler at offset 0 is the original entry point byte for byte."""
    bins, c1, c2, K = 1001, 400, 433, 18
    ca, cb, exp = make_case(eng, bins, c1, c2, K, 1, seed=7)
    dist = real_distance(eng, ca, cb, c1, c2, 1, exp)
    seed, P = 12345, 96

    def fused(lo, hi, p0, n, k=None):
        k = torch.zeros(hi - lo, dtype=torch.int32, device="cuda") if k is None else k
        return eng.permutation_exceedances_s1(ca[lo:hi].contiguous(), cb[lo:hi].contiguous(), c1, c2, seed, p0, n,
                                              c1 + c2, lo, exp, c1, c2, dist[lo:hi].contiguous(), k)

    whole = fused(0, bins, 0, P).cpu().numpy()
    split = np.concatenate([fused(0, 333, 0, P).cpu().numpy(), fused(333, bins, 0, P).cpu().numpy()])
    assert whole.tolist() == split.tolist()
    k = fused(0, bins, 0, 40)
    k = fused(0, bins, 40, 5, k)
    k = fused(0, bins, 45, P - 45, k)
    assert whole.tolist() == k.cpu().numpy().tolist()
    oa, ob = eng.shuffled_counts_philox(ca, cb, c1, c2, seed, nperm=3, width=c1 + c2, bin_offset=9)
    ra, rb = eng.shuffled_counts_philox_range(ca, cb, c1, c2, seed, 0, 3, c1 + c2, bin_offset=9)
    assert torch.equal(oa, ra) and torch.equal(ob, rb)
    ta, tb = eng.shuffled_counts_philox_range(ca, cb, c1, c2, seed, 2, 1, c1 + c2, bin_offset=9)
    assert torch.equal(ta[0], oa[2]) and torch.equal(tb[0], ob[2])


def test_null_exceedances_against_numpy(eng):
    bins, c1, c2, K, P = 700, 60, 67, 15, 9
    ca, cb, exp = make_case(eng, bins, c1, c2, K, 1, seed=3)
    dist = real_distance(eng, ca, cb, c1, c2, 1, exp)
    oa, ob = eng.shuffled_counts_philox_range(ca, cb, c1, c2, 5, 0, P, c1 + c2)
    sa = eng.scores_s1(oa.reshape(-1, K), c1, exp).reshape(P, bins, K)
    sb = eng.scores_s1(ob.reshape(-1, K), c2, exp).reshape(P, bins, K)
    k = eng.null_exceedances(sa, sb, dist, torch.full((bins,), 3, dtype=torch.int32, device="cuda")).cpu().numpy()
    d = (sa - sb).cpu().numpy()
    null = (np.sum(d * d, axis=2) * np.sign(np.sum(d, axis=2))).astype(np.float32)
    want = 3 + (np.abs(null) >= np.abs(dist.cpu().numpy())).sum(axis=0)
    assert k.tolist() == want.tolist()


def test_null_hypothesis_and_planted_differences(eng):
    """Both groups i.i.d. from one label distribution: P(p <= 0.05) stays within a binomial tolerance of 0.05.  Bins where
    the groups hold different single states: every shuffle mixes them, so k = 0 and p = 1 / (P + 1)."""
    from epilogos_b200.backend import CudaBackend
    bins, c1, c2, K, P, planted = 6000, 50, 50, 18, 99, 200
    rng = np.random.default_rng(11)
    probs = rng.dirichlet(np.ones(K))
    x = rng.choice(K, size=(bins, c1 + c2), p=probs).astype(np.int8)
    x[:planted, :c1] = 0
    x[:planted, c1:] = 1
    ca = eng.bin_counts(eng.pack_states(np.ascontiguousarray(x[:, :c1])).cuda(), c1, K)
    cb = eng.bin_counts(eng.pack_states(np.ascontiguousarray(x[:, c1:])).cuda(), c2, K)
    n1, _ = eng.expected_tables((ca + cb).contiguous(), c1 + c2, want_s2=False)
    exp = eng.normalize(n1)
    dist = real_distance(eng, ca, cb, c1, c2, 1, exp)
    k = CudaBackend().permutation_exceedances(ca, cb, dist, P, 77, c1, c2, c1 + c2, 0, 1, exp, (c1, c2),
                                              (0, 0)).cpu().numpy().view(np.uint32)
    p = (k + 1.0) / (P + 1.0)
    assert np.all(k[:planted] == 0) and np.all(p[:planted] == 1.0 / (P + 1))
    h0 = p[planted:]
    n = len(h0)
    assert np.mean(h0 <= 0.05) <= 0.05 + 3.0 * np.sqrt(0.05 * 0.95 / n)
    assert np.mean(h0 <= 0.5) > 0.3                       # not degenerate: the null is not always far away


def test_cli_end_to_end_and_permutation_zero_is_the_runs_null(eng, tmp_path, monkeypatch):
    """Steps 1-3 with the temp files kept: permutation 0 of the counts is the run's own null; then the CLI with and
    without --null-permutations writes the same other files."""
    from click.testing import CliRunner
    from epilogos_b200 import expected, expectedCombination, helpers, run, scores, session
    from test_cli import META
    from test_host_stages import write_tsv
    rng = np.random.default_rng(5)
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    for chrom, rows in (("chr1", 900), ("chr2", 611)):
        x = rng.integers(0, 18, size=(rows, 127)).astype(np.int8)
        x[: rows // 4, :60] = rng.integers(0, 3, size=(rows // 4, 60))
        write_tsv(a / ("m_%s.txt.gz" % chrom), x[:, :60], chrom=chrom, gz=True)
        write_tsv(b / ("m_%s.txt.gz" % chrom), x[:, 60:], chrom=chrom, gz=True)
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    monkeypatch.setenv("EPILOGOS_B200_SEED", "19")

    out = tmp_path / "steps"; out.mkdir()
    session.clear()
    fa, fb = a / "m_chr1.txt.gz", b / "m_chr1.txt.gz"
    expected.main(fa, fb, 18, 1, out, "t", 1, False)
    expectedCombination.main(out, out / "exp_freq_t.npy", "t", False)
    scores.main(fa, fb, 18, 1, out, out / "exp_freq_t.npy", "t", 1, 17, -1, False, permutations=1)
    null = np.load(out / "temp_nullDistances_t_m_chr1.npz")["nullDistances"]
    k = np.load(out / "temp_permutations_t_m_chr1.npz")["exceedances"]
    loc, delta = helpers.read_scores(out / "pairwiseDelta_t_m_chr1.txt.gz")
    dist, _ = eng.pairwise_real_reduce(torch.from_numpy(delta.astype(np.float32)).cuda(), False)
    assert k.tolist() == (np.abs(null) >= np.abs(dist.cpu().numpy())).astype(np.uint32).tolist()
    session.clear()

    def cli(outdir, *extra):
        session.clear()
        r = CliRunner().invoke(run.main, ["-m", "paired", "-a", str(a), "-b", str(b), "-o", str(outdir), "-j", str(meta),
                                          "-s", "1", "-n", "-t", "3", "-z", "500"] + list(extra))
        session.clear()
        assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)

    plain, perm = tmp_path / "plain", tmp_path / "perm"
    cli(plain)
    cli(perm, "--null-permutations", "200")
    rows = gzip.open(perm / "pairwisePermutation_a_b_s1.txt.gz", "rt").read().splitlines()
    assert len(rows) == 900 + 611 and all(len(r.split("\t")) == 6 for r in rows)
    kk = np.array([int(r.split("\t")[3]) for r in rows])
    assert kk.min() == 0 and kk.max() <= 200
    assert sorted(p.name for p in plain.iterdir()) == sorted(p.name for p in perm.iterdir() if "Permutation" not in p.name)
    for f in plain.iterdir():
        g = perm / f.name
        if f.name.endswith(".gz"):
            assert gzip.open(f).read() == gzip.open(g).read(), f.name
        else:
            assert f.read_bytes() == g.read_bytes(), f.name
