"""Multi-group kernels (csrc/multigroup.cu): the G-way sampler against the two-group sampler and its marginal laws, the
statistic against the numpy oracle, the fused S1 counts against the composed path, the S2 composed counts against numpy
under two workspace caps, and the p-values under the null and with planted differences."""
import numpy as np
import pytest

import multigroup_oracle as mgo

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


def split(width, parts):
    base, extra = divmod(width, parts)
    return [base + (1 if g >= parts - extra else 0) for g in range(parts)]


def make_case(eng, bins, sizes, K, saliency, seed, planted=0, quiet=0):
    """Counts [G, bins, K] of disjoint column ranges of one labelled matrix (a share of bins differs between groups), the
    union's expected table, and the union's counts.  The first `planted` bins give group g the single state g % K; the
    next `quiet` bins are all state 0."""
    rng = np.random.default_rng(seed)
    G, N = len(sizes), sum(sizes)
    probs = rng.dirichlet(np.ones(K) * 0.3, size=4)
    kind = rng.integers(0, 4, size=bins)
    cols = np.concatenate([[g] * n for g, n in enumerate(sizes)])
    shift = rng.random((bins, G)) < 0.3
    x = np.empty((bins, N), dtype=np.int8)
    for b in range(bins):
        for g in range(G):
            lo = int(np.sum(sizes[:g]))
            x[b, lo:lo + sizes[g]] = rng.choice(K, size=sizes[g], p=probs[(kind[b] + shift[b, g]) % 4])
    for b in range(planted):
        x[b] = cols % K
    x[planted:planted + quiet] = 0
    offs = np.concatenate([[0], np.cumsum(sizes)])
    groups = [list(range(offs[g], offs[g + 1])) for g in range(G)]
    cnt = eng.group_counts(eng.pack_states(x).cuda(), N, K, groups)
    union = cnt.sum(dim=0, dtype=torch.int32).to(torch.int16).contiguous()
    n1, n2 = eng.expected_tables(union, N, want_s1=saliency == 1, want_s2=saliency == 2)
    exp = eng.normalize(n1 if saliency == 1 else n2)
    return cnt, exp, union


def group_scores(eng, cnt, sizes, saliency, exp):
    out = []
    for g, n in enumerate(sizes):
        c = cnt[g].contiguous().clone()
        out.append(eng.scores_s1(c, n, exp) if saliency == 1 else eng.scores_s2(c, n, exp, perms=n * (n - 1)))
    return torch.stack(out)


def test_two_groups_draw_as_the_paired_sampler(eng):
    for bins, sizes, K, off in [(1001, [400, 433], 18, 0), (777, [60, 67], 15, (1 << 33) + 5)]:
        cnt, _, _ = make_case(eng, bins, sizes, K, 1, seed=bins)
        want_a, want_b = eng.shuffled_counts_philox_range(cnt[0].contiguous(), cnt[1].contiguous(), sizes[0], sizes[1],
                                                          99, 3, 5, sum(sizes), bin_offset=off)
        got = eng.multigroup_shuffled_counts_range(cnt, sizes, 99, 3, 5, bin_offset=off)
        assert torch.equal(got[:, 0], want_a) and torch.equal(got[:, 1], want_b)


@pytest.mark.parametrize("G", [3, 8, 64])
def test_every_draw_keeps_state_totals_and_group_sizes(eng, G):
    sizes = split(13 * G + 5, G)
    bins, K, P = 301, 18, 6
    cnt, _, union = make_case(eng, bins, sizes, K, 1, seed=G, planted=3, quiet=2)
    out = eng.multigroup_shuffled_counts_range(cnt, sizes, 7, 0, P, bin_offset=11).cpu().numpy().astype(np.int64)
    u = union.cpu().numpy().astype(np.int64)
    assert np.array_equal(out.sum(axis=1), np.broadcast_to(u, (P, bins, K)))
    assert np.array_equal(out.sum(axis=3), np.broadcast_to(np.array(sizes)[None, :, None], (P, G, bins)))
    assert (out >= 0).all()


def test_group_margins_are_hypergeometric(eng):
    """At 10^6 draws of one bin, group g's count of a state follows hypergeom(N, c_s, n_g) whatever g's place in the
    draw order: the first, a middle and the last group."""
    from scipy import stats
    sizes, K, P = [7, 19, 12, 25, 9], 15, 1_000_000
    N = sum(sizes)
    labels = np.repeat(np.arange(K), split(N, K))
    rng = np.random.default_rng(5)
    x = rng.permutation(labels).astype(np.int8)[None, :]
    offs = np.concatenate([[0], np.cumsum(sizes)])
    groups = [list(range(offs[g], offs[g + 1])) for g in range(len(sizes))]
    cnt = eng.group_counts(eng.pack_states(x).cuda(), N, K, groups)
    out = eng.multigroup_shuffled_counts_range(cnt, sizes, 2024, 0, P)
    c = np.bincount(labels, minlength=K)
    for g, s in [(0, 2), (2, 7), (len(sizes) - 1, 13)]:
        obs = np.bincount(out[:, g, 0, s].cpu().numpy().astype(np.int64), minlength=c[s] + 1)
        pmf = stats.hypergeom(N, c[s], sizes[g]).pmf(np.arange(len(obs)))
        keep = pmf * P >= 5
        o = np.append(obs[keep], obs[~keep].sum())
        e = np.append(pmf[keep] * P, P - (pmf[keep] * P).sum())
        assert stats.chisquare(o, e * o.sum() / e.sum()).pvalue > 1e-4, (g, s)


@pytest.mark.parametrize("K", [15, 18, 25])
@pytest.mark.parametrize("width,parts", [(127, 5), (833, 3), (833, 8)])
def test_stat_against_the_oracle(eng, K, width, parts):
    sizes = split(width, parts)
    for saliency in (1, 2):
        cnt, exp, _ = make_case(eng, 613, sizes, K, saliency, seed=width + K + parts, planted=5, quiet=4)
        sc = group_scores(eng, cnt, sizes, saliency, exp)
        t, g, s, sign = eng.multigroup_stat(sc, sizes)
        wt, wg, ws, wsign = mgo.stat_and_driver(sc.cpu().numpy(), sizes)
        assert t.cpu().numpy().view(np.uint64).tolist() == wt.view(np.uint64).tolist()
        assert g.cpu().numpy().tolist() == wg.tolist() and s.cpu().numpy().tolist() == ws.tolist()
        assert sign.cpu().numpy().tolist() == wsign.tolist()
        assert np.all(wt[5:9] == 0.0) and wt[9:].max() > 0


def test_two_groups_is_the_paired_distance(eng):
    """G = 2: T N^2 / (n1 n2) = sum_s (S_A[s] - S_B[s])^2."""
    sizes = [400, 433]
    cnt, exp, _ = make_case(eng, 1001, sizes, 18, 1, seed=1)
    sc = group_scores(eng, cnt, sizes, 1, exp)
    t = eng.multigroup_stat(sc, sizes)[0].cpu().numpy()
    d = (sc[0] - sc[1]).double().cpu().numpy()
    want = (d * d).sum(axis=1)
    N = sum(sizes)
    np.testing.assert_allclose(t * N * N / (sizes[0] * sizes[1]), want, rtol=1e-6, atol=1e-30)


def composed_k(eng, cnt, sizes, seed, bin_offset, nperm, saliency, exp, t):
    """k from the sampler and the score entry points, counted by the oracle."""
    out = eng.multigroup_shuffled_counts_range(cnt, sizes, seed, 0, nperm, bin_offset=bin_offset)
    null = torch.stack([group_scores(eng, out[p], sizes, saliency, exp) for p in range(nperm)])
    return mgo.exceedances(null.cpu().numpy(), sizes, t.cpu().numpy()), null


CASES = [  # bins, sizes, K, nperm, bin_offset
    (1001, split(833, 4), 18, 64, 0),
    (777, split(127, 5), 15, 7, 12345),
    (513, split(833, 2), 18, 1, 5),
    (301, split(127, 3), 18, 33, (1 << 33) + 1),
    (99, split(833, 8), 25, 7, (1 << 32) + 7),
]


@pytest.mark.parametrize("case", CASES)
def test_fused_s1_equals_the_composed_path(eng, case):
    bins, sizes, K, nperm, off = case
    cnt, exp, _ = make_case(eng, bins, sizes, K, 1, seed=bins + K)
    t = eng.multigroup_stat(group_scores(eng, cnt, sizes, 1, exp), sizes)[0]
    want, null = composed_k(eng, cnt, sizes, 31337, off, nperm, 1, exp, t)
    assert eng.multigroup_s1_fused_fits(sizes, K)
    fused = eng.multigroup_exceedances_s1(cnt, sizes, 31337, 0, nperm, off, exp, t,
                                          torch.zeros(bins, dtype=torch.int32, device="cuda"))
    assert fused.cpu().numpy().tolist() == want.tolist(), case
    k = torch.full((bins,), 2, dtype=torch.int32, device="cuda")
    k = eng.multigroup_null_exceedances(null.contiguous(), sizes, t, k)
    assert (k.cpu().numpy() - 2).tolist() == want.tolist()
    assert want.max() <= nperm and (want.sum() > 0 or nperm == 1)


def test_fused_s1_splits_and_batches(eng):
    bins, sizes, K, P = 1001, split(833, 4), 18, 96
    cnt, exp, _ = make_case(eng, bins, sizes, K, 1, seed=7)
    t = eng.multigroup_stat(group_scores(eng, cnt, sizes, 1, exp), sizes)[0]

    def fused(lo, hi, p0, n, k=None):
        k = torch.zeros(hi - lo, dtype=torch.int32, device="cuda") if k is None else k
        return eng.multigroup_exceedances_s1(cnt[:, lo:hi], sizes, 5, p0, n, lo, exp, t[lo:hi].contiguous(), k)

    whole = fused(0, bins, 0, P).cpu().numpy()
    parts = np.concatenate([fused(0, 333, 0, P).cpu().numpy(), fused(333, bins, 0, P).cpu().numpy()])
    assert whole.tolist() == parts.tolist()
    k = fused(0, bins, 0, 40)
    k = fused(0, bins, 40, 5, k)
    k = fused(0, bins, 45, P - 45, k)
    assert whole.tolist() == k.cpu().numpy().tolist()


@pytest.mark.parametrize("sizes", [split(127, 3), split(833, 5)])
def test_s2_composed_against_numpy_under_two_caps(eng, sizes):
    from epilogos_b200.backend import CudaBackend
    bins, K, P = 257, 15, 9
    cnt, exp, _ = make_case(eng, bins, sizes, K, 2, seed=len(sizes))
    be = CudaBackend()
    t, g, s, sign = be.multigroup_stat(cnt, sizes, 2, exp, workspace_bytes=4 * len(sizes) * K * 50)
    wt = mgo.stat_and_driver(group_scores(eng, cnt, sizes, 2, exp).cpu().numpy(), sizes)[0]
    assert t.cpu().numpy().view(np.uint64).tolist() == wt.view(np.uint64).tolist()
    want, _ = composed_k(eng, cnt, sizes, 4242, 17, P, 2, exp, t)
    for cap in (1 << 30, 6 * len(sizes) * K * 100):
        got = be.multigroup_exceedances(cnt, sizes, t, P, 4242, 17, 2, exp, workspace_bytes=cap)
        assert got.cpu().numpy().tolist() == want.tolist(), cap


@pytest.mark.parametrize("saliency", [1, 2])
def test_null_hypothesis_planted_and_quiet_bins(eng, saliency):
    """Groups i.i.d. from one label distribution: P(p <= 0.05) within a binomial tolerance of 0.05.  Bins where every group
    holds its own single state: every shuffle mixes them, so p = 1 / (P + 1).  Bins of one state: T = 0 and p = 1."""
    from epilogos_b200.backend import CudaBackend
    sizes, bins, K, P, planted, quiet = [20, 30, 25, 25], 5000, 18, 99, 150, 50
    N = sum(sizes)
    rng = np.random.default_rng(11)
    x = rng.choice(K, size=(bins, N), p=rng.dirichlet(np.ones(K))).astype(np.int8)
    cols = np.concatenate([[g] * n for g, n in enumerate(sizes)])
    x[:planted] = cols
    x[planted:planted + quiet] = 0
    offs = np.concatenate([[0], np.cumsum(sizes)])
    cnt = eng.group_counts(eng.pack_states(x).cuda(), N, K, [list(range(offs[g], offs[g + 1])) for g in range(4)])
    union = cnt.sum(dim=0, dtype=torch.int32).to(torch.int16).contiguous()
    n1, n2 = eng.expected_tables(union, N, want_s1=saliency == 1, want_s2=saliency == 2)
    exp = eng.normalize(n1 if saliency == 1 else n2)
    be = CudaBackend()
    t = be.multigroup_stat(cnt, sizes, saliency, exp)[0]
    k = be.multigroup_exceedances(cnt, sizes, t, P, 77, 0, saliency, exp).cpu().numpy().view(np.uint32)
    p = mgo.pvalues(k, P)
    assert np.all(p[:planted] == 1.0 / (P + 1))
    assert np.all(t.cpu().numpy()[planted:planted + quiet] == 0.0) and np.all(p[planted:planted + quiet] == 1.0)
    h0 = p[planted + quiet:]
    tol = 3.0 * np.sqrt(0.05 * 0.95 / len(h0))
    assert abs(np.mean(h0 <= 0.05) - 0.05) <= tol
    assert np.mean(h0 <= 0.5) > 0.3


def test_cli_end_to_end_against_the_library(eng, tmp_path, monkeypatch):
    """--multigroup on the CUDA backend, S1 (fused) and S2 (composed): every line of multigroupMetrics against the backend
    routes called on the same counts with the run's file seeds."""
    import gzip
    from click.testing import CliRunner
    from epilogos_b200 import run, session
    from epilogos_b200.backend import CudaBackend
    from epilogos_b200.pairwise import file_seed
    from test_cli import META
    from test_host_stages import write_tsv
    monkeypatch.setenv("EPILOGOS_B200_SEED", "4242")
    rng = np.random.default_rng(3)
    K, C = 18, 60
    inp = tmp_path / "in"
    inp.mkdir()
    mats = {}
    for chrom, rows in (("chr1", 1500), ("chr2", 900)):
        x = rng.integers(0, K, size=(rows, C), dtype=np.int8)
        x[rng.random(rows) < 0.3] = K - 1
        x[:200, :20] = rng.integers(0, 3, size=(200, 20))
        write_tsv(inp / ("epilogos_matrix_%s.txt.gz" % chrom), x, chrom=chrom, gz=True)
        mats[chrom] = x
    (tmp_path / "g.tsv").write_text("A\t1-20\nB\t21-45\nC\t46-60\n")
    (tmp_path / "meta.tsv").write_text(META)
    sizes = [20, 25, 15]
    offs = [0, 20, 45, 60]
    be = CudaBackend()
    for saliency in (1, 2):
        out = tmp_path / ("out%d" % saliency)
        session.clear()
        r = CliRunner().invoke(run.main, ["-m", "paired", "-i", str(inp), "-o", str(out), "-j", str(tmp_path / "meta.tsv"),
                                          "--groups", str(tmp_path / "g.tsv"), "--multigroup", "A,B,C", "-s",
                                          str(saliency), "--null-permutations", "50"])
        session.clear()
        assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)
        lines = gzip.open(out / "A_B_C" / ("multigroupMetrics_A_B_C_s%d.txt.gz" % saliency), "rt").read().splitlines()
        tables, cnts = [], {}
        for chrom, x in mats.items():
            cnt = eng.group_counts(eng.pack_states(x).cuda(), C, K, [list(range(offs[g], offs[g + 1])) for g in range(3)])
            union = cnt.sum(dim=0, dtype=torch.int32).to(torch.int16).contiguous()
            n1, n2 = eng.expected_tables(union, C, want_s1=saliency == 1, want_s2=saliency == 2)
            tables.append(n1 if saliency == 1 else n2)
            cnts[chrom] = cnt
        exp = eng.normalize(sum(tables))
        want_t, want_k = [], []
        for chrom in ("chr1", "chr2"):
            t, g, s, sign = be.multigroup_stat(cnts[chrom], sizes, saliency, exp)
            k = be.multigroup_exceedances(cnts[chrom], sizes, t, 50, file_seed(4242, "epilogos_matrix_" + chrom), 0,
                                          saliency, exp)
            want_t += ["%.5e" % v for v in t.cpu().numpy()]
            want_k += [str(v) for v in k.cpu().numpy().view(np.uint32)]
        assert [ln.split("\t")[3] for ln in lines] == want_t
        assert [ln.split("\t")[7] for ln in lines] == want_k
        assert (out / "A_B_C" / ("regionsOfInterest_A_B_C_s%d.txt" % saliency)).exists()
