"""Paired statistics stage (epilogos_b200.roi_pairwise): the oracle's definitions, and the paired command line end to
end on a stand-in backend that answers the statistics with scipy.  The kernels themselves are covered by
test_pairwise_stats_gpu.py."""
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.special
import scipy.stats
import torch
from click.testing import CliRunner

from fake_backend import OracleBackend
from oracle import epilogos_oracle as orc
from oracle import pairwise_stats_oracle as pso
from test_cli import META
from test_host_stages import ROOT, write_tsv


class StatsBackend(OracleBackend):
    """OracleBackend plus the paired statistics, answered with numpy / scipy (the subsamples come from numpy's generator,
    not from the device's keyed permutation)."""

    def pairwise_real_reduce(self, delta, text_round_trip=True):
        d, md = orc.paired_real_reductions(np.asarray(delta, dtype=np.float32), text_round_trip)
        return torch.from_numpy(np.asarray(d, dtype=np.float32)), torch.from_numpy(md.astype(np.int32))

    def null_pool(self, null_dist, quiescent):
        return torch.from_numpy(pso.null_pool([null_dist.numpy()], [quiescent.numpy()]))

    def null_subsample(self, pool, trials, size, seed):
        n = pool.numel()
        idx = np.stack([np.random.default_rng([int(seed) & (2 ** 63 - 1), t]).permutation(n)[:size]
                        for t in range(trials)]).astype(np.int32)
        return torch.from_numpy(idx), torch.from_numpy(pool.numpy()[idx])

    def gennorm_fit(self, samples):
        params = np.array([pso.fit(row) for row in samples.numpy()], dtype=np.float64)
        return params, np.tile(np.array([[1, 1]], dtype=np.int32), (len(params), 1))

    def gennorm_pvalues(self, x, beta, loc, scale):
        return torch.from_numpy(pso.pvalues_gammaincc(x.numpy(), beta, loc, scale))

    def bh_adjust(self, p):
        return torch.from_numpy(pso.bh(p.numpy()))


def bh_brute_force(p):
    """q_i = min(1, min over p_j >= p_i of p_j * n / #{k : p_k <= p_j})."""
    p = np.asarray(p, dtype=np.float64)
    n = len(p)
    rank = np.array([np.sum(p <= v) for v in p])
    return np.array([min(1.0, min(p[j] * n / rank[j] for j in range(n) if p[j] >= v)) for v in p])


def test_bh_oracle_matches_the_definition_with_ties_zeros_and_ones():
    rng = np.random.default_rng(3)
    for n in (1, 2, 7, 300):
        p = rng.random(n) ** 3
        p[rng.random(n) < 0.2] = 0.0
        p[rng.random(n) < 0.2] = 1.0
        if n > 4:
            p[1:4] = p[0]                                       # ties
            p[rng.random(n) < 0.3] = np.round(p[rng.random(n) < 0.3].mean(), 2) if n > 10 else p[0]
        np.testing.assert_allclose(pso.bh(p), bh_brute_force(p), rtol=1e-14, atol=0)
    # the result does not depend on the order of tied values
    p = np.array([0.01, 0.04, 0.04, 0.04, 0.5, 0.0, 1.0, 0.04])
    q = pso.bh(p)
    perm = rng.permutation(len(p))
    assert pso.bh(p[perm]).tobytes() == q[perm].tobytes()


def test_pvalue_identity_gammaincc_equals_two_sided_gennorm():
    rng = np.random.default_rng(4)
    for beta in (0.1, 0.4, 1.0, 2.0, 5.0, 10.0):
        x = (scipy.stats.gennorm.rvs(beta, size=400, random_state=rng) * 1.7 + 0.3).astype(np.float32)
        a = pso.pvalues_gammaincc(x, beta, 0.3, 1.7)
        b = pso.pvalues(x, beta, 0.3, 1.7)
        ok = b > 1e-300
        np.testing.assert_allclose(a[ok], b[ok], rtol=1e-10)
        assert np.all((a >= 0) & (a <= 1))
    assert pso.pvalues_gammaincc(np.float32([0.5]), 0.7, 0.5, 2.0)[0] == 1.0
    assert scipy.special.gammaincc(2.0, np.inf) == 0.0


def make_paired_inputs(tmp_path, golden, chroms=("chr1", "chr2")):
    g = golden("paired_synth_c30_c25_k18")
    xa, xb = g["xa"], g["xb"]
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    parts = np.array_split(np.arange(len(xa)), len(chroms))
    for chrom, rows in zip(chroms, parts):
        name = "epilogos_matrix_%s.txt.gz" % chrom
        write_tsv(a / name, xa[rows], chrom=chrom, gz=True)
        write_tsv(b / name, xb[rows], chrom=chrom, gz=True)
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    return a, b, meta


def run_paired_cli(monkeypatch, a, b, meta, out, *extra):
    from epilogos_b200 import run, session
    session.clear()
    monkeypatch.setattr(session, "_backend", StatsBackend())
    r = CliRunner().invoke(run.main, ["-m", "paired", "-a", str(a), "-b", str(b), "-o", str(out), "-j", str(meta),
                                      "-s", "1", "-w", "9"] + list(extra))
    assert r.exit_code == 0, r.output + repr(r.exception)
    session.clear()
    return r.output


def read_gz(path):
    with gzip.open(path, "rt") as f:
        return f.read()


def test_paired_cli_writes_metrics_and_regions(tmp_path, golden, monkeypatch):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "77")
    a, b, meta = make_paired_inputs(tmp_path, golden, chroms=("chr10", "chr2", "chr1"))
    names = ["S%d" % i for i in range(1, 19)]
    out = tmp_path / "out"
    log = run_paired_cli(monkeypatch, a, b, meta, out, "-n", "-t", "5", "-z", "200", "-d")
    assert "STEP 4" in log and "not built" in log
    tag = "a_b_s1"
    assert not list(out.glob("temp_*")) and not (out / ("exp_freq_%s.npy" % tag)).exists()
    assert sorted(p.name for p in out.glob("pairwiseDelta_*")) == ["pairwiseDelta_%s_epilogos_matrix_%s.txt.gz" % (tag, c)
                                                                   for c in ("chr1", "chr10", "chr2")]
    metrics = read_gz(out / ("pairwiseMetrics_%s.txt.gz" % tag)).splitlines()
    rows = [l.split("\t") for l in metrics]
    assert all(len(r) == 8 for r in rows)
    # chromosome order: numbered chromosomes ascending
    assert [r[0] for r in rows] == sorted((r[0] for r in rows), key=lambda c: int(c[3:]))
    # the first six columns against the oracle on the deltas as written
    want = []
    for c in ("chr1", "chr2", "chr10"):
        txt = read_gz(out / ("pairwiseDelta_%s_epilogos_matrix_%s.txt.gz" % (tag, c))).splitlines()
        cols = [l.split("\t") for l in txt]
        delta = np.array([[float(v) for v in l[3:]] for l in cols], dtype=np.float64).astype(np.float32)
        d, md = orc.paired_real_reductions(delta, round_trip=False)
        want.append(pso.metrics_text([l[0] for l in cols], [int(l[1]) for l in cols], [int(l[2]) for l in cols], names,
                                     md, d))
    assert ["\t".join(r[:6]) for r in rows] == "".join(want).splitlines()
    p = np.array([float(r[6]) for r in rows])
    q = np.array([float(r[7]) for r in rows])
    assert np.all((p >= 0) & (p <= 1)) and np.all((q >= 0) & (q <= 1)) and np.all(q >= p * (1 - 1e-5))
    roi = (out / ("regionsOfInterest_%s.txt" % tag)).read_text().splitlines()
    assert roi and all(len(l.split("\t")) == 8 for l in roi)

    # without -n: six columns, no fit
    out6 = tmp_path / "out6"
    run_paired_cli(monkeypatch, a, b, meta, out6)
    m6 = read_gz(out6 / ("pairwiseMetrics_%s.txt.gz" % tag)).splitlines()
    assert [l.split("\t") for l in m6] == [r[:6] for r in rows]
    assert all(len(l.split("\t")) == 6 for l in (out6 / ("regionsOfInterest_%s.txt" % tag)).read_text().splitlines())
    assert not list(out6.glob("temp_*"))


def test_paired_statistics_from_files_equal_the_in_process_hand_over(tmp_path, golden, monkeypatch):
    """EPILOGOS_B200_KEEP_TEMP=1 makes the score stage write its temp files and step 4 read them (and the deltas from
    pairwiseDelta text); the outputs are the same bytes as with the in-memory hand-over."""
    monkeypatch.setenv("EPILOGOS_B200_SEED", "5")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    mem, disk = tmp_path / "mem", tmp_path / "disk"
    run_paired_cli(monkeypatch, a, b, meta, mem, "-n", "-t", "3", "-z", "150")
    monkeypatch.setenv("EPILOGOS_B200_KEEP_TEMP", "1")
    run_paired_cli(monkeypatch, a, b, meta, disk, "-n", "-t", "3", "-z", "150")
    for name in ("pairwiseMetrics_a_b_s1.txt.gz", "regionsOfInterest_a_b_s1.txt"):
        assert (mem / name).read_bytes() == (disk / name).read_bytes()
    assert not list(disk.glob("temp_*"))


def test_paired_statistics_main_returns_the_median_fit(tmp_path, golden, monkeypatch):
    """roi_pairwise.main on the files of steps 1-3: the returned fit is the median-NLL trial of scipy fits on the
    subsamples, and the p / BH columns are those of the oracle with these parameters."""
    from epilogos_b200 import expected, expectedCombination, roi_pairwise, scores, session
    a, b, meta = make_paired_inputs(tmp_path, golden, chroms=("chr1",))
    out = tmp_path / "out"; out.mkdir()
    be = StatsBackend()
    session.clear()
    fa, fb = a / "epilogos_matrix_chr1.txt.gz", b / "epilogos_matrix_chr1.txt.gz"
    expected.main(fa, fb, 18, 1, out, "t", 1, False, backend=be)
    expectedCombination.main(out, out / "exp_freq_t.npy", "t", False, backend=be)
    monkeypatch.setenv("EPILOGOS_B200_SEED", "11")
    scores.main(fa, fb, 18, 1, out, out / "exp_freq_t.npy", "t", 1, 17, -1, False, backend=be)
    null = np.load(out / "temp_nullDistances_t_epilogos_matrix_chr1.npz")["nullDistances"]
    quies = np.load(out / "temp_quiescence_t_epilogos_matrix_chr1.npz")["quiescenceArr"]
    res = roi_pairwise.main(out, meta, "t", out / "exp_freq_t.npy", 9, True, 5, 120, backend=be, seed=11)
    tab = res["trials"]
    pool = pso.null_pool([null], [quies])
    assert tab["pool_size"] == len(pool) and len(tab["nll"]) == 5
    assert tab["chosen"] == pso.median_trial(tab["nll"])
    assert (res["beta"], res["loc"], res["scale"]) == (tab["beta"][tab["chosen"]], tab["loc"][tab["chosen"]],
                                                       tab["scale"][tab["chosen"]])
    rows = [l.split("\t") for l in read_gz(out / "pairwiseMetrics_t.txt.gz").splitlines()]
    delta = np.array([[float(v) for v in l.split("\t")[3:]] for l in
                      read_gz(out / "pairwiseDelta_t_epilogos_matrix_chr1.txt.gz").splitlines()]).astype(np.float32)
    d, md = orc.paired_real_reductions(delta, round_trip=False)
    p = pso.pvalues_gammaincc(d, res["beta"], res["loc"], res["scale"])
    want = pso.metrics_text([r[0] for r in rows], [int(r[1]) for r in rows], [int(r[2]) for r in rows],
                            ["S%d" % i for i in range(1, 19)], md, d, p, pso.bh(p))
    assert "\n".join("\t".join(r) for r in rows) + "\n" == want
    roi = (out / "regionsOfInterest_t.txt").read_text()
    assert roi == pso.roi_text([r[0] for r in rows], [int(r[1]) for r in rows], [int(r[2]) for r in rows],
                               ["S%d" % i for i in range(1, 19)], md, d, 9, p, pso.bh(p))
    assert not list(out.glob("temp_*")) and not (out / "exp_freq_t.npy").exists()
    session.clear()


def test_paired_statistics_need_three_null_values(tmp_path, golden, monkeypatch):
    from epilogos_b200 import roi_pairwise
    be = StatsBackend()
    chunks = [dict(null=torch.zeros(4), quiescence=torch.tensor([1, 1, 0, 1], dtype=torch.uint8))]
    with pytest.raises(ValueError, match="at least 3"):
        roi_pairwise.fit_null(be, chunks, 5, 100, 1)


GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
os.environ["EPILOGOS_B200_SHARD"] = {shard!r}
os.environ["EPILOGOS_B200_SEED"] = "31"
import torch.distributed as td
from pathlib import Path
from test_pairwise_stats import StatsBackend
from epilogos_b200 import dist, run
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
out = Path({out!r}); a = Path({a!r}); b = Path({b!r})
pairs = [(f, b / f.name) for f in sorted(a.glob("*"))]
say = (lambda *x, **k: print(*x, **k, flush=True)) if dist.rank() == 0 else (lambda *x, **k: None)
run.run_stages(pairs, "paired", 18, 1, out, "a_b_s1", out / "exp_freq_a_b_s1.npy", 1, 17, -1, {meta!r}, 9, False, say,
               backend=StatsBackend(), pvalBool=True, numTrials=3, samplingSize=150)
td.destroy_process_group()
"""


@pytest.mark.parametrize("shard", ["rows", "files"])
def test_two_gloo_ranks_write_the_same_statistics_as_one(tmp_path, golden, monkeypatch, shard):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "31")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    one = tmp_path / "one"
    run_paired_cli(monkeypatch, a, b, meta, one, "-n", "-t", "3", "-z", "150", "-w", "9")
    two = tmp_path / "two"; two.mkdir()
    port = 34500 + (os.getpid() % 2000) + (7 if shard == "files" else 0)
    code = GLOO_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), shard=shard, port=port, out=str(two), a=str(a),
                              b=str(b), meta=str(meta))
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    assert read_gz(one / "pairwiseMetrics_a_b_s1.txt.gz") == read_gz(two / "pairwiseMetrics_a_b_s1.txt.gz")
    assert (one / "regionsOfInterest_a_b_s1.txt").read_text() == (two / "regionsOfInterest_a_b_s1.txt").read_text()
    assert not list(two.glob("temp_*"))
