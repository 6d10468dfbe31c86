"""Paired statistics kernels (csrc/pairwise_stats.cu) against scipy / the numpy restatements of
oracle/pairwise_stats_oracle.py, and paired step 4 end to end on the CUDA backend."""
import gzip
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import scipy.special
import scipy.stats

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import epilogos_oracle as orc            # noqa: E402
from oracle import pairwise_stats_oracle as pso      # noqa: E402

PARAM_TOL = 2e-4        # the optimizer's xatol is 1e-4
NLL_RTOL = 1e-9


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import build, engine
    build.build()
    engine.device_info()
    return engine


def check_fit(params, status, points, what):
    beta, loc, scale, nll = pso.fit(points)
    got = params
    assert abs(got[0] - beta) <= PARAM_TOL and abs(got[1] - loc) <= PARAM_TOL and abs(got[2] - scale) <= PARAM_TOL, \
        "%s: device %r, scipy %r" % (what, tuple(got[:3]), (beta, loc, scale))
    assert abs(got[3] - nll) <= NLL_RTOL * abs(nll), "%s: NLL %r vs %r" % (what, got[3], nll)


def test_pvalues_against_gammaincc(eng):
    rows = []
    for beta in np.linspace(0.1, 10.0, 12):
        z = np.concatenate(([0.0], np.logspace(-12, np.log10(800.0), 400)))
        rows.append((beta, (z ** (1.0 / beta)).astype(np.float32)))
    for beta, x in rows:
        for loc, scale in ((0.0, 1.0), (0.25, 3.0)):
            xs = (x.astype(np.float64) * scale + loc).astype(np.float32)
            got = eng.gennorm_pvalues(torch.from_numpy(xs).cuda(), beta, loc, scale).cpu().numpy()
            want = scipy.special.gammaincc(1.0 / beta, (np.abs(xs.astype(np.float64) - loc) / scale) ** beta)
            big = want > 1e-300
            rel = np.abs(got[big] - want[big]) / want[big]
            assert rel.max() <= 1e-12, "beta=%g: max relative error %g" % (beta, rel.max())
            assert np.all(np.abs(got[~big]) <= 2e-300)
            assert got[xs == np.float32(loc)].tolist() == [1.0] * int(np.sum(xs == np.float32(loc)))
    far = eng.gennorm_pvalues(torch.tensor([1e30, -1e30], dtype=torch.float32).cuda(), 2.0, 0.0, 1.0).cpu().numpy()
    assert far.tolist() == [0.0, 0.0]


@pytest.mark.parametrize("n", [1, 4097, 1 << 20, 15_500_000])
def test_bh_is_bitwise_the_numpy_restatement(eng, n):
    rng = np.random.default_rng(n)
    p = rng.random(n) ** 4
    p[rng.random(n) < 0.05] = 0.0
    p[rng.random(n) < 0.05] = 1.0
    if n > 100:
        p[rng.integers(0, n, n // 10)] = p[rng.integers(0, n, n // 10)]       # ties
        p[: n // 50] = np.round(p[: n // 50], 3)
    got = eng.bh_adjust(torch.from_numpy(p).cuda()).cpu().numpy()
    want = pso.bh(p)
    assert got.tobytes() == want.tobytes(), "%d of %d differ" % (int(np.sum(got != want)), n)


def test_subsample_indices(eng):
    n, trials, size = 1_234_567, 16, 100_000
    pool = torch.arange(n, dtype=torch.float32).cuda()
    idx, samples = eng.null_subsample(pool, trials, size, 99)
    idx2, _ = eng.null_subsample(pool, trials, size, 99)
    idx3, _ = eng.null_subsample(pool, trials, size, 100)
    a = idx.cpu().numpy()
    assert np.array_equal(a, idx2.cpu().numpy()) and not np.array_equal(a, idx3.cpu().numpy())
    assert a.min() >= 0 and a.max() < n
    assert np.array_equal(samples.cpu().numpy(), a.astype(np.float32))
    for t in range(trials):
        assert len(np.unique(a[t])) == size
    assert not np.array_equal(a[0], a[1])
    counts = np.bincount((a.ravel().astype(np.int64) * 200) // n, minlength=200)
    chi2 = scipy.stats.chisquare(counts)
    assert chi2.pvalue > 1e-4, chi2
    # a pool no larger than the subsample: the trial is a permutation of the whole pool
    whole, _ = eng.null_subsample(pool[:1000], 1, 1000, 5)
    assert sorted(whole.cpu().numpy()[0].tolist()) == list(range(1000))


@pytest.mark.parametrize("beta", [0.4, 1.0, 2.0, 5.0])
def test_fit_matches_scipy_on_gennorm_samples(eng, beta):
    rng = np.random.default_rng(int(beta * 10))
    x = (scipy.stats.gennorm.rvs(beta, size=(3, 5000), random_state=rng) * 2.5 - 0.7).astype(np.float32)
    params, status = eng.gennorm_fit(torch.from_numpy(x).cuda())
    params = params.cpu().numpy()
    again = eng.gennorm_fit(torch.from_numpy(x).cuda())[0].cpu().numpy()
    assert params.tobytes() == again.tobytes()
    for t in range(3):
        check_fit(params[t], status[t], x[t], "beta=%g trial %d" % (beta, t))


def synthetic_null(eng, bins=20000):
    xa = orc.synth_states(bins, 12, 18, seed=41)
    xb = orc.synth_states(bins, 9, 18, seed=42)
    r = eng.paired_host(eng.pack_states(xa), 12, eng.pack_states(xb), 9, 18, 1, 17, seed=1234)
    return r["null"][0], r["quiescent"]


@pytest.mark.parametrize("source", ["paired_real10_k18", "paired_synth_c30_c25_k18", "synthetic"])
def test_fit_on_null_distances_and_median_trial(eng, golden, source):
    if source == "synthetic":
        null, q = synthetic_null(eng)
    else:
        g = golden(source)
        null, q = g["s1_null"], g["s1_quiescence"]
    pool = eng.null_compact(torch.from_numpy(np.ascontiguousarray(null)).cuda(),
                            torch.from_numpy(q.astype(np.uint8)).cuda()).cpu().numpy()
    assert pool.tobytes() == null[~q].tobytes()
    n = len(pool)
    trials, size = (11, 5000) if n > 5000 else (1, n)
    idx, samples = eng.null_subsample(torch.from_numpy(pool).cuda(), trials, size, 2024)
    params, status = eng.gennorm_fit(samples)
    params, idx = params.cpu().numpy(), idx.cpu().numpy()
    want = pso.fit_trials(pool, idx)
    for t in range(trials):
        check_fit(params[t], status[t], pool[idx[t]], "%s trial %d" % (source, t))
    assert pso.median_trial(params[:, 3]) == pso.median_trial(want[:, 3])


def test_null_compact_with_permutations(eng):
    rng = np.random.default_rng(8)
    null = rng.standard_normal((3, 70001)).astype(np.float32)
    q = rng.random(70001) < 0.4
    pool = eng.null_compact(torch.from_numpy(null).cuda(), torch.from_numpy(q.astype(np.uint8)).cuda()).cpu().numpy()
    assert pool.tobytes() == pso.null_pool([null], [q]).tobytes()


def run_steps_1_to_3(tmp_path, g, saliency):
    from test_host_stages import run_paired_pipeline
    run_paired_pipeline(tmp_path, g["xa"], g["xb"], int(g["num_states"]), saliency, None, int(g["seed"]),
                        int(g["group_size"]), int(g["quiescent_state"]))
    meta = tmp_path / "meta.tsv"
    meta.write_text("zero_index\tone_index\tshort_name\tlong_name\n" +
                    "".join("%d\t%d\tS%d\tstate %d\n" % (i, i + 1, i + 1, i + 1) for i in range(int(g["num_states"]))))
    return tmp_path / "out", meta


@pytest.mark.parametrize("name", ["paired_real10_k18", "paired_synth_c30_c25_k18"])
def test_paired_step4_end_to_end_on_the_device(eng, golden, tmp_path, name, monkeypatch):
    """Seeded reference-mode steps 1-3, then step 4 on the CUDA backend: the pool is the golden's non-quiescent null,
    the fit is scipy's on that pool, the text is the oracle's with the device's parameters; `python -m` on a copy of the
    same directory writes the same files."""
    from epilogos_b200 import roi_pairwise, session
    g = golden(name)
    out, meta = run_steps_1_to_3(tmp_path, g, 1)
    names = ["S%d" % i for i in range(1, int(g["num_states"]) + 1)]
    tag = "a_b_s1"
    copy = tmp_path / "copy"
    shutil.copytree(out, copy)
    with gzip.open(out / ("pairwiseDelta_%s_epilogos_matrix_chr1.txt.gz" % tag), "rt") as f:
        lines = [l.split("\t") for l in f.read().splitlines()]
    session.clear()
    res = roi_pairwise.main(out, meta, tag, out / ("exp_freq_%s.npy" % tag), 125, True, 101, 100000, seed=3)
    null, q = g["s1_null"], g["s1_quiescence"]
    pool = null[~q]
    tab = res["trials"]
    assert tab["pool_size"] == len(pool) and len(tab["nll"]) == 1       # N <= S: one fit on the whole pool
    beta, loc, scale, nll = pso.fit(pool)
    assert abs(res["beta"] - beta) <= PARAM_TOL and abs(res["loc"] - loc) <= PARAM_TOL
    assert abs(res["scale"] - scale) <= PARAM_TOL and abs(tab["nll"][0] - nll) <= NLL_RTOL * abs(nll)
    delta = np.array([[float(v) for v in l[3:]] for l in lines]).astype(np.float32)
    d, md = orc.paired_real_reductions(delta, round_trip=False)
    p = pso.pvalues_gammaincc(d, res["beta"], res["loc"], res["scale"])
    chrom, st, en = [l[0] for l in lines], [int(l[1]) for l in lines], [int(l[2]) for l in lines]
    with gzip.open(out / ("pairwiseMetrics_%s.txt.gz" % tag), "rt") as f:
        got = f.read()
    want = pso.metrics_text(chrom, st, en, names, md, d, p, pso.bh(p))
    assert got == want
    assert (out / ("regionsOfInterest_%s.txt" % tag)).read_text() == pso.roi_text(chrom, st, en, names, md, d, 125, p,
                                                                                   pso.bh(p))
    assert not list(out.glob("temp_*"))
    env = dict(os.environ, EPILOGOS_B200_SEED="3")
    r = subprocess.run([sys.executable, "-m", "epilogos_b200.roi_pairwise", str(copy), str(meta), tag,
                        str(copy / ("exp_freq_%s.npy" % tag)), "125", "True"], env=env, capture_output=True, text=True,
                       cwd=str(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    assert r.returncode == 0, r.stdout + r.stderr
    for f in ("pairwiseMetrics_%s.txt.gz" % tag, "regionsOfInterest_%s.txt" % tag):
        assert (copy / f).read_bytes() == (out / f).read_bytes()


def test_paired_cli_on_the_device_hand_over_equals_files(tmp_path, golden, monkeypatch):
    """The paired command with -n on the CUDA backend (device null, N > S): the in-memory hand-over and the route through
    the temp files give the same bytes, and a second run with the same seed repeats them."""
    from click.testing import CliRunner
    from epilogos_b200 import run, session
    from test_host_stages import write_tsv
    xa = orc.synth_states(30000, 12, 18, seed=51)
    xb = orc.synth_states(30000, 9, 18, seed=52)
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    for chrom, sl in (("chr1", slice(0, 18000)), ("chr2", slice(18000, 30000))):
        write_tsv(a / ("m_%s.txt.gz" % chrom), xa[sl], chrom=chrom, gz=True)
        write_tsv(b / ("m_%s.txt.gz" % chrom), xb[sl], chrom=chrom, gz=True)
    meta = tmp_path / "meta.tsv"
    meta.write_text("zero_index\tone_index\tshort_name\tlong_name\n" +
                    "".join("%d\t%d\tS%d\tstate %d\n" % (i, i + 1, i + 1, i + 1) for i in range(18)))
    monkeypatch.setenv("EPILOGOS_B200_SEED", "808")
    outs = []
    for i, keep in enumerate(("", "", "1")):
        if keep:
            monkeypatch.setenv("EPILOGOS_B200_KEEP_TEMP", keep)
        out = tmp_path / ("out%d" % i)
        session.clear()
        r = CliRunner().invoke(run.main, ["-m", "paired", "-a", str(a), "-b", str(b), "-o", str(out), "-j", str(meta),
                                          "-s", "2", "-n", "-t", "11", "-z", "5000"])
        assert r.exit_code == 0, r.output + repr(r.exception)
        assert not list(out.glob("temp_*")) and not list(out.glob("exp_freq_*"))
        outs.append(out)
    session.clear()
    for f in ("pairwiseMetrics_a_b_s2.txt.gz", "regionsOfInterest_a_b_s2.txt"):
        assert (outs[0] / f).read_bytes() == (outs[1] / f).read_bytes() == (outs[2] / f).read_bytes()
    with gzip.open(outs[0] / "pairwiseMetrics_a_b_s2.txt.gz", "rt") as fh:
        rows = [l.split("\t") for l in fh.read().splitlines()]
    assert len(rows) == 30000 and all(len(r) == 8 for r in rows)


def test_two_gpus_write_the_same_files_as_one(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from test_host_stages import write_tsv
    xa = orc.synth_states(20000, 10, 18, seed=61)
    xb = orc.synth_states(20000, 8, 18, seed=62)
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    write_tsv(a / "m_chr1.txt.gz", xa, gz=True)
    write_tsv(b / "m_chr1.txt.gz", xb, gz=True)
    meta = tmp_path / "meta.tsv"
    meta.write_text("zero_index\tone_index\tshort_name\tlong_name\n" +
                    "".join("%d\t%d\tS%d\tstate %d\n" % (i, i + 1, i + 1, i + 1) for i in range(18)))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, EPILOGOS_B200_SEED="17")
    outs = []
    for n in (1, 2):
        out = tmp_path / ("out%d" % n)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", str(n), "--master-port",
               str(29600 + n), "-m", "epilogos_b200.run", "-m", "paired", "-a", str(a), "-b", str(b), "-o", str(out),
               "-j", str(meta), "-n", "-t", "11", "-z", "5000"]
        r = subprocess.run(cmd, env=env, cwd=root, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout + r.stderr
        outs.append(out)
    for f in ("pairwiseMetrics_a_b_s1.txt.gz", "regionsOfInterest_a_b_s1.txt"):
        assert (outs[0] / f).read_bytes() == (outs[1] / f).read_bytes()
