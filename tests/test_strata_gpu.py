"""The stratified sampler and the fused stratified S1 kernel on the device (csrc/strata.cu): one stratum equals the
unstratified samplers byte for byte; draws equal the numpy restatement (tests/strata_oracle.py) outside a 1e-8 CDF margin
(as test_sampler_gpu.py compares them); the draws of A' fit the exact convolution of the per-stratum multivariate
hypergeometrics; the fused kernel equals the composed path; a one-stratum CLI run equals the run without strata; and a
stratified test keeps its level where tissue, not group, drives the states."""
import types

import numpy as np
import pytest

import strata_oracle as sto
from oracle import epilogos_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

MARGIN = 1e-8
MAX_EXCLUDED = 10
SEED_HI = 0x5EA7A7A000000000


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


def counts_of(x, K):
    return orc.bin_counts(x, K).astype(np.int64)


def max_width(H, G):
    """The widest stratum whose sampler tables, sizes and need counts fit the kernel's 200 KB."""
    return ((200 * 1024 - G * 256 * 4 - H * G * 4) // 8 - 3) // 2


def strata_rows(sizes, K, bins, seed):
    """(cnt_h [H, rows, K], per-group counts [G, rows, K]) of a synthetic matrix whose columns are the strata one after
    the other, each stratum's columns group after group."""
    N = int(np.sum(sizes))
    x = orc.synth_states(bins, N, K, seed).astype(np.int64)
    x[: bins // 8] = np.random.default_rng(seed).integers(0, K, size=(bins // 8, N))
    cnt_h, per_group = [], [np.zeros((bins, K), dtype=np.int64) for _ in sizes[0]]
    at = 0
    for row in sizes:
        w = int(sum(row))
        cnt_h.append(counts_of(x[:, at:at + w], K))
        for g, n in enumerate(row):
            per_group[g] += counts_of(x[:, at:at + n], K) if n else 0
            at += n
    return np.stack(cnt_h), np.stack(per_group)


# ---- one stratum is the unstratified draw ---------------------------------------------------------------------------------

@pytest.mark.parametrize("case", [((400, 433), 18, 2000, 0, 33, 0), ((60, 67), 15, 700, (1 << 32) - 4, 4, (1 << 33) + 3),
                                  ((40, 50, 37), 18, 900, 5, 9, 12345), (tuple([13] * 64), 25, 200, (1 << 32) - 1, 1, 7)],
                         ids=lambda c: "G%d_N%d" % (len(c[0]), sum(c[0])))
def test_one_stratum_equals_the_unstratified_samplers(eng, case):
    sizes, K, bins, p0, P, off = case
    cnt_h, cnt_g = strata_rows([list(sizes)], K, bins, seed=sum(sizes))
    seed = SEED_HI | sum(sizes)
    got = host(eng.stratified_shuffled_counts_range(dev16(cnt_h), [list(sizes)], seed, p0, P, bin_offset=off))
    if len(sizes) == 2:
        oa, ob = eng.shuffled_counts_philox_range(dev16(cnt_g[0]), dev16(cnt_g[1]), sizes[0], sizes[1], seed, p0, P,
                                                  sum(sizes), bin_offset=off)
        want = np.stack([host(oa), host(ob)], axis=1)
    else:
        want = host(eng.multigroup_shuffled_counts_range(dev16(cnt_g), list(sizes), seed, p0, P, bin_offset=off))
    assert got.shape == want.shape and np.array_equal(got, want)


# ---- draw for draw against the restatement ---------------------------------------------------------------------------------

DRAWS = [  # sizes [H][G], K, bins, perm_offset, nperm, bin_offset
    ([[200, 200], [200, 233]], 18, 600, 0, 16, 0),                                     # 833 biosamples
    ([[10, 5, 3], [0, 7, 0], [1, 0, 0], [4, 4, 4], [0, 0, 1]], 15, 800, (1 << 32) - 8, 8, (1 << 33) + 3),
    ([[6, 7]] * 63 + [[1, 0]], 18, 300, 3, 8, 77),
    ([[3, 0, 2]] * 32 + [[0, 1, 1]] * 32, 12, 300, 0, 8, 0),
    ([[max_width(2, 2) - 3000, 3000], [50, 60]], 18, 40, 0, 4, 5),                      # the sampler's width limit
    ([[max_width(2, 3) - 200, 100, 100], [1, 1, 1]], 18, 40, (1 << 32) - 4, 4, 0),
]


@pytest.mark.parametrize("case", DRAWS, ids=lambda c: "H%d_G%d_N%d" % (len(c[0]), len(c[0][0]), np.sum(c[0])))
def test_draws_equal_the_restatement(eng, case):
    sizes, K, bins, p0, P, off = case
    cnt_h, _ = strata_rows(sizes, K, bins, seed=int(np.sum(sizes)))
    H, rows, _ = cnt_h.shape
    G = len(sizes[0])
    seed = SEED_HI | int(np.sum(sizes)) * 64 + H
    got = host(eng.stratified_shuffled_counts_range(dev16(cnt_h), sizes, seed, p0, P, bin_offset=off))
    got = got.transpose(0, 2, 1, 3).reshape(P * rows, G, K)
    r = sto.draw_stratified_shuffle(seed, p0 + np.repeat(np.arange(P, dtype=np.int64), rows),
                                    off + np.tile(np.arange(rows, dtype=np.int64), P), np.tile(cnt_h, (1, P, 1)), sizes)
    far = r["margin"] > MARGIN
    bad = far[:, None, None] & (r["x"] != got)
    assert not bad.any(), "%d outcomes differ, first at %s" % (bad.sum(), np.argwhere(bad)[0])
    print("stratified %s: %d draws compared, %d inside the margin" % (case[1:], far.sum(), (~far).sum()))
    assert (~far).sum() <= MAX_EXCLUDED
    # every stratum keeps its make-up: the groups' totals are the sums of their sizes
    assert np.array_equal(got.sum(axis=2), np.tile(np.sum(sizes, axis=0), (P * rows, 1)))
    assert np.array_equal(got.sum(axis=1), np.tile(cnt_h.sum(axis=0), (P, 1)))


def test_a_stratum_beyond_the_width_limit_is_refused(eng):
    cnt = torch.zeros((2, 1, 4), dtype=torch.int16, device="cuda")
    with pytest.raises(Exception, match="too wide"):
        eng.stratified_shuffled_counts_range(cnt, [[max_width(2, 2) - 100, 101], [1, 1]], 1, 0, 1)


# ---- goodness of fit -------------------------------------------------------------------------------------------------------

def mvhg_pmf(comb, n):
    """{counts tuple: probability} of the multivariate hypergeometric draw of n labels from the state counts comb."""
    from itertools import product
    from math import comb as C
    total = C(int(sum(comb)), n)
    out = {}
    for a in product(*[range(c + 1) for c in comb]):
        if sum(a) == n:
            out[a] = np.prod([C(int(c), int(v)) for c, v in zip(comb, a)]) / total
    return out


def test_goodness_of_fit_against_the_exact_convolution(eng):
    """K = 3; stratum 0: 3 + 3 biosamples with state counts (2, 3, 1), stratum 1: 2 + 4 with (1, 2, 3).  A' is the sum of
    two independent multivariate hypergeometric draws; 10^6 draws against its exact distribution.  The chi-square
    threshold is the 1e-6 upper quantile of chi-square at its degrees of freedom (15 outcomes - 1 = 14): 54.6.  Seed
    fixed."""
    from scipy.stats import chi2
    sizes = [[3, 3], [2, 4]]
    cnt_h = np.array([[[2, 3, 1]], [[1, 2, 3]]], dtype=np.int64).repeat(125000, axis=1)
    out = host(eng.stratified_shuffled_counts_range(dev16(cnt_h), sizes, 0x5EED0F17, 0, 8))
    a = out[:, 0].reshape(-1, 3)
    assert len(a) == 10 ** 6
    exact = {}
    for x0, p0 in mvhg_pmf((2, 3, 1), 3).items():
        for x1, p1 in mvhg_pmf((1, 2, 3), 2).items():
            key = tuple(u + v for u, v in zip(x0, x1))
            exact[key] = exact.get(key, 0.0) + p0 * p1
    assert abs(sum(exact.values()) - 1.0) < 1e-12 and len(exact) == 15
    keys = sorted(exact)
    code = {k: i for i, k in enumerate(keys)}
    seen = np.bincount([code[tuple(r)] for r in map(tuple, a)], minlength=len(keys))
    expected = np.array([exact[k] for k in keys]) * len(a)
    stat = float(((seen - expected) ** 2 / expected).sum())
    threshold = 54.6
    assert abs(chi2.isf(1e-6, len(keys) - 1) - threshold) < 0.1
    print("chi-square %.2f over %d outcomes (threshold %.1f)" % (stat, len(keys), threshold))
    assert stat < threshold


# ---- the fused kernel equals the composed path ---------------------------------------------------------------------------

def composed_counts(eng, cnt_h, sizes, cnt_a, cnt_b, seed, p0, P, off, exp, wa, wb, dist):
    k = torch.zeros(cnt_a.shape[0], dtype=torch.int32, device="cuda")
    out = eng.stratified_shuffled_counts_range(cnt_h, sizes, seed, p0, P, bin_offset=off)
    rows, K = cnt_a.shape
    sa = eng.scores_s1(out[:, 0].contiguous().reshape(-1, K), wa, exp).reshape(P, rows, K)
    sb = eng.scores_s1(out[:, 1].contiguous().reshape(-1, K), wb, exp).reshape(P, rows, K)
    return eng.null_exceedances(sa, sb, dist, k)


@pytest.mark.parametrize("P", [1, 7, 8, 31, 32, 1000])
@pytest.mark.parametrize("where", ["smem", "l1"])
def test_fused_s1_equals_the_composed_path(eng, P, where):
    sizes = [[30, 25], [12, 40], [8, 0], [0, 5]] if where == "smem" else [[400, 400], [420, 380]]
    K = 18
    bins = 3000 if P < 1000 else 400
    cnt_h, cnt_g = strata_rows(sizes, K, bins, seed=P + len(sizes))
    wa, wb = int(np.sum(sizes, axis=0)[0]), int(np.sum(sizes, axis=0)[1])
    union = cnt_g.sum(axis=0)
    exp = torch.from_numpy(orc.normalize_expected(union.sum(axis=0)).astype(np.float32)).cuda()
    ca, cb = dev16(cnt_g[0]), dev16(cnt_g[1])
    delta, _ = eng.pairwise_combine(eng.scores_s1(ca, wa, exp), eng.scores_s1(cb, wb, exp))
    dist, _ = eng.pairwise_real_reduce(delta, True)
    seed, p0, off = SEED_HI | P, ((1 << 32) - P - 3) if P < 32 else 11, (1 << 33) + 5
    h = dev16(cnt_h)
    k = torch.zeros(bins, dtype=torch.int32, device="cuda")
    fused = eng.stratified_exceedances_s1(h, sizes, ca, cb, seed, p0, P, off, exp, wa, wb, dist, k)
    want = composed_counts(eng, h, sizes, ca, cb, seed, p0, P, off, exp, wa, wb, dist)
    assert torch.equal(fused, want)
    kk = fused.cpu().numpy()
    assert kk.min() >= 0 and kk.max() <= P and (P < 8 or (kk.min() < P and kk.max() > 0))


def test_fused_s1_with_one_stratum_equals_the_unstratified_kernel(eng):
    K, sizes = 18, [[400, 433]]
    cnt_h, cnt_g = strata_rows(sizes, K, 2000, seed=5)
    exp = torch.from_numpy(orc.normalize_expected(cnt_g.sum(axis=0).sum(axis=0)).astype(np.float32)).cuda()
    ca, cb = dev16(cnt_g[0]), dev16(cnt_g[1])
    delta, _ = eng.pairwise_combine(eng.scores_s1(ca, 400, exp), eng.scores_s1(cb, 433, exp))
    dist, _ = eng.pairwise_real_reduce(delta, True)
    k1 = torch.zeros(2000, dtype=torch.int32, device="cuda")
    k2 = torch.zeros(2000, dtype=torch.int32, device="cuda")
    eng.stratified_exceedances_s1(dev16(cnt_h), sizes, ca, cb, 77, 3, 100, 9, exp, 400, 433, dist, k1)
    eng.permutation_exceedances_s1(ca, cb, 400, 433, 77, 3, 100, 833, 9, exp, 400, 433, dist, k2)
    assert torch.equal(k1, k2)


# ---- the command line ------------------------------------------------------------------------------------------------------

def test_one_stratum_cli_run_equals_the_run_without_strata(tmp_path, monkeypatch, golden):
    from click.testing import CliRunner
    from epilogos_b200 import run, session
    from test_groups import assert_same_outputs
    from test_pairwise_stats import make_paired_inputs
    monkeypatch.setenv("EPILOGOS_B200_SEED", "2024")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    strata = tmp_path / "strata.tsv"
    strata.write_text("all\t1-55\n")
    for saliency in (1, 2):
        common = ["-m", "paired", "-a", a, "-b", b, "-j", meta, "-s", saliency, "-w", 9, "-n", "-t", 5, "-z", 500,
                  "--null-permutations", 40, "--roi-permutations", 6]
        for name, extra in (("plain", []), ("strata", ["--strata", strata])):
            session.clear()
            r = CliRunner().invoke(run.main, [str(v) for v in common + ["-o", tmp_path / ("%s%d" % (name, saliency))]
                                              + extra])
            assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)
        session.clear()
        assert_same_outputs(tmp_path / ("strata%d" % saliency), tmp_path / ("plain%d" % saliency))


# ---- the property the feature exists for --------------------------------------------------------------------------------

def test_strata_keep_the_level_where_tissue_drives_the_states(eng):
    """Two tissues; a bin's dominant state depends only on the tissue (each label is the tissue's state with probability
    0.7, else uniform over 18 states), never on the group.  A holds 40 biosamples of tissue X and 10 of Y, B the reverse.
    P = 199, so a valid test has P(p <= 0.05) <= 10/200 = 0.05 per bin, and the 20,000 independent bins give a count of
    at most Binomial(20000, 0.05): mean 1000, sd 30.8.  With strata the share must stay below 0.05 + 5 sd / 20000 =
    0.0577; a free shuffle mixes the tissues and must exceed 0.3 (it is near 1 here).  Seeds fixed: deterministic."""
    from epilogos_b200.backend import CudaBackend
    be = CudaBackend()
    K, bins, P = 18, 20000, 199
    rng = np.random.default_rng(20261022)
    dom = rng.integers(0, K, size=(bins, 2))
    tissue_a = np.array([0] * 40 + [1] * 10)
    tissue_b = np.array([0] * 10 + [1] * 40)

    def labels(tissue):
        x = dom[:, tissue]
        noise = rng.random(x.shape) >= 0.7
        return np.where(noise, rng.integers(0, K, size=x.shape), x)
    xa, xb = labels(tissue_a), labels(tissue_b)
    x = np.concatenate([xa, xb], axis=1)
    ca, cb = dev16(counts_of(xa, K)), dev16(counts_of(xb, K))
    exp = torch.from_numpy(orc.normalize_expected(counts_of(x, K).sum(axis=0)).astype(np.float32)).cuda()
    delta, _ = eng.pairwise_combine(eng.scores_s1(ca, 50, exp), eng.scores_s1(cb, 50, exp))
    dist, _ = eng.pairwise_real_reduce(delta, True)
    tissue = np.concatenate([tissue_a, tissue_b])
    columns = [np.flatnonzero(tissue == t) for t in (0, 1)]
    strata = types.SimpleNamespace(sizes=[[40, 10], [10, 40]],
                                   counts=dev16(np.stack([counts_of(x[:, c], K) for c in columns])))
    shares = {}
    for name, extra in (("free", {}), ("strata", {"strata": strata})):
        k = be.permutation_exceedances(ca, cb, dist, P, 99, 50, 50, 100, 0, 1, exp, (50, 50), (50 * 49, 50 * 49),
                                       **extra).cpu().numpy().view(np.uint32)
        shares[name] = float(np.mean((1.0 + k) / (P + 1.0) <= 0.05))
    print("share of bins with p <= 0.05: %s" % shares)
    assert shares["strata"] <= 0.0577
    assert shares["free"] > 0.3
