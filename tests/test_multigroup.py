"""The multi-group statistic's definition (tests/multigroup_oracle.py) and the fused kernel's shape query, on the CPU.  The
kernels are covered by test_multigroup_gpu.py."""
import numpy as np

import multigroup_oracle as mgo
import sampler_oracle as so


def scores(rng, G, bins, K):
    return rng.normal(size=(G, bins, K)).astype(np.float32)


def test_two_groups_is_the_squared_score_distance():
    rng = np.random.default_rng(1)
    sizes = [400, 433]
    sc = scores(rng, 2, 500, 18)
    t, _ = mgo.statistic(sc, sizes)
    d = sc[0].astype(np.float64) - sc[1].astype(np.float64)
    N = sum(sizes)
    np.testing.assert_allclose(t * N * N / (sizes[0] * sizes[1]), (d * d).sum(axis=1), rtol=1e-12)


def test_equal_scores_give_exactly_zero():
    rng = np.random.default_rng(2)
    for sizes in ([1, 65534], [25, 25, 25, 26, 26], list(range(1, 65))):
        one = scores(rng, 1, 100, 25)
        t, m = mgo.statistic(np.repeat(one, len(sizes), axis=0), sizes)
        assert np.all(t == 0.0) and np.array_equal(m, one[0].T.astype(np.float64))
        k = mgo.exceedances(np.repeat(one, len(sizes), axis=0)[None].repeat(3, axis=0), sizes, t)
        assert np.all(k == 3) and np.all(mgo.pvalues(k, 3) == 1.0)


def test_driver_is_the_group_and_state_furthest_from_the_mean():
    sizes = [10, 20, 30]
    sc = np.zeros((3, 4, 5), dtype=np.float32)
    sc[1, 0, 3] = -2.0                                # bin 0: group 1 low in state 3
    sc[2, 1, 0] = 1.0                                 # bin 1: group 2 high in state 0
    sc[0, 3, 1] = sc[0, 3, 2] = 1.0                   # bin 3: a tie between states 1 and 2 -> the first
    t, g, s, sign = mgo.stat_and_driver(sc, sizes)
    assert (g[0], s[0], sign[0]) == (1, 3, -1)
    assert (g[1], s[1], sign[1]) == (2, 0, 1)
    assert t[2] == 0.0 and (g[2], s[2], sign[2]) == (0, 0, 1)       # all equal: the first group and state
    assert (g[3], s[3], sign[3]) == (0, 1, 1)
    assert np.all(t[[0, 1, 3]] > 0)


def test_fused_kernel_shape_query():
    """The fused S1 kernel takes groups up to the S1 value table's width whose tables fit in shared memory; the library
    answers without a device."""
    from epilogos_b200 import engine
    assert engine.multigroup_s1_fused_fits([104] * 7 + [105], 18)
    assert engine.multigroup_s1_fused_fits([13] * 64, 18)
    assert engine.multigroup_s1_fused_fits([400, 433], 32)
    assert not engine.multigroup_s1_fused_fits([4096, 10], 18)             # wider than the S1 value table
    assert not engine.multigroup_s1_fused_fits([3000, 3000], 18)           # tables beyond shared memory
    assert not engine.multigroup_s1_fused_fits([833], 18)                  # one group is no comparison


# ---- the command line on a stand-in backend ------------------------------------------------------------------------------

import gzip  # noqa: E402
import os  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402

import pytest  # noqa: E402
import torch  # noqa: E402
from click.testing import CliRunner  # noqa: E402

from oracle import epilogos_oracle as orc  # noqa: E402
from oracle import pairwise_stats_oracle as pso  # noqa: E402
from test_groups import K, assert_same_outputs, make_inputs  # noqa: E402
from test_host_stages import ROOT  # noqa: E402
from test_permutations import PermBackend  # noqa: E402

MGROUPS = """g1\t1-5
g2\t6-10
g3\t11-15
g4\t16-20
g5\t21-24
a\t1-8
all\t1-24
"""
MCOLS = {"g1": range(0, 5), "g2": range(5, 10), "g3": range(10, 15), "g4": range(15, 20), "g5": range(20, 24),
         "a": range(0, 8)}
STATE_NAMES = ["S%d" % i for i in range(1, K + 1)]


def draw_exceedances(cnt, sizes, t, nperm, seed, bin_offset, saliency, exp, score):
    """k per bin from the device's G-way draws (sampler_oracle.draw_multigroup_shuffle): permutation p of row r from the
    stream keyed by (seed, p, GLOBAL bin bin_offset + r)."""
    G, rows, k = cnt.shape
    comb = cnt.sum(axis=0)
    x = so.draw_multigroup_shuffle(seed, np.repeat(np.arange(nperm), rows), bin_offset + np.tile(np.arange(rows), nperm),
                                   np.tile(comb, (nperm, 1)), sizes)["x"].reshape(nperm, rows, G, k)
    null = np.stack([np.stack([score(x[p, :, g], n) for g, n in enumerate(sizes)]) for p in range(nperm)])
    return mgo.exceedances(null.astype(np.float32), sizes, np.asarray(t))


class MultiBackend(PermBackend):
    """The stand-in plus the multi-group routes: its own scores, the numpy definitions and numpy G-way draws."""

    def _score_fn(self, saliency, exp):
        e = exp.numpy()
        if saliency == 1:
            return lambda c, n: orc.s1_scores_from_counts(c, n, e)
        return lambda c, n: orc.s2_scores_from_counts(c, n * (n - 1), e)

    def multigroup_stat(self, cnt, sizes, saliency, exp, exact=False, workspace_bytes=None):
        c = cnt.numpy().view(np.uint16).astype(np.int64)
        score = self._score_fn(saliency, exp)
        sc = np.stack([score(c[g], n) for g, n in enumerate(sizes)]).astype(np.float32)
        t, g, s, sign = mgo.stat_and_driver(sc, sizes)
        return (torch.from_numpy(t), torch.from_numpy(g.astype(np.uint8)), torch.from_numpy(s.astype(np.uint8)),
                torch.from_numpy(sign.astype(np.int8)))

    def multigroup_exceedances(self, cnt, sizes, t, nperm, seed, bin_offset, saliency, exp, exact=False,
                               workspace_bytes=None):
        c = cnt.numpy().view(np.uint16).astype(np.int64)
        k = draw_exceedances(c, sizes, t.numpy(), nperm, seed, bin_offset, saliency, exp, self._score_fn(saliency, exp))
        return torch.from_numpy(k.astype(np.uint32).view(np.int32))


def run_cli(monkeypatch, *args, backend=None):
    from epilogos_b200 import run, session
    session.clear()
    monkeypatch.setattr(session, "_backend", backend or MultiBackend())
    r = CliRunner().invoke(run.main, [str(a) for a in args])
    session.clear()
    return r


def ok(r):
    assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)


def inputs(tmp_path):
    inp, _, meta, data = make_inputs(tmp_path)
    gfile = tmp_path / "mgroups.tsv"
    gfile.write_text(MGROUPS)
    return inp, gfile, meta, data


def test_flag_rules_and_their_precedence(tmp_path, monkeypatch):
    inp, gfile, meta, _ = inputs(tmp_path)
    out = tmp_path / "out"
    base = ["-m", "paired", "-i", inp, "-o", out, "-j", meta, "--groups", gfile]
    cases = [
        (["-m", "paired", "-a", inp, "-b", inp, "-o", out, "-j", meta, "--multigroup", "g1,g2"],
         "ERROR: [--multigroup] requires [--groups]"),
        (["-i", inp, "-o", out, "-j", meta, "--groups", gfile, "--multigroup", "g1,g2"],
         "ERROR: [--multigroup] requires [-m, --mode] 'paired'"),
        (base + ["--multigroup", "g1,zz"], "ERROR: [--multigroup] group 'zz' is not defined in the group file"),
        (base + ["--multigroup", "g1,g2,g1"], "ERROR: [--multigroup] 'g1,g2,g1' lists group 'g1' twice"),
        (base + ["--multigroup", "g1"], "ERROR: [--multigroup] 'g1' names fewer than 2 groups"),
        (base + ["--multigroup", "g2,a,g3"], "ERROR: [--multigroup] groups 'g2' and 'a' share biosample 6"),
        (base + ["--multigroup", "g1,g2", "-n"], "ERROR: [--multigroup] not compatible with [-n, --null-distribution] flag"),
        (base + ["--multigroup", "g1,g2", "-g", 3], "ERROR: [--multigroup] not compatible with [-g, --group-size] option"),
        # the order among the new rules, and after every existing rule
        (base + ["--multigroup", "g1", "--multigroup", "g1,zz"],
         "ERROR: [--multigroup] group 'zz' is not defined in the group file"),
        (base + ["--multigroup", "g1,g1", "--multigroup", "g2"], "ERROR: [--multigroup] 'g1,g1' lists group 'g1' twice"),
        (base + ["--multigroup", "g2,a", "--multigroup", "g3"], "ERROR: [--multigroup] 'g3' names fewer than 2 groups"),
        (base + ["--multigroup", "g1,a", "-n"], "ERROR: [--multigroup] groups 'g1' and 'a' share biosample 1"),
        (base + ["--multigroup", "g1,zz", "--null-permutations", 0],
         "ERROR: Number of null permutations must be between 1 and 1000000"),
        (base + ["--multigroup", "g1,zz", "-t", 0], "ERROR: Number of trials must be greater than zero"),
        (["-m", "paired", "-i", inp, "-j", meta, "--groups", gfile, "--multigroup", "g1"],
         "ERROR: [-o, --output-directory] required"),
        # paired --groups with neither --compare nor --multigroup keeps its message
        (base, "ERROR: [-m, --mode] 'paired' with [--groups] requires at least one [--compare]"),
    ]
    for args, message in cases:
        r = run_cli(monkeypatch, *args)
        assert r.output.strip().splitlines()[-1] == message, (args, r.output)
        assert not list(out.glob("*/multigroup*"))


def expected_outputs(data, sizes_cols, saliency, P, seed, roi_width):
    """multigroupMetrics and regionsOfInterest text from numpy: counts, background, scores, the statistic and the draws."""
    from epilogos_b200.pairwise import file_seed
    from epilogos_b200.roi import max_mean, orderChromosomes
    names = list(sizes_cols)
    cols = [np.asarray(sizes_cols[n]) for n in names]
    sizes = [len(c) for c in cols]
    per_file = {}
    tables = []
    for fname, (chrom, x) in data.items():
        cnt = np.stack([orc.bin_counts(x[:, c], K) for c in cols]).astype(np.int64)
        union = cnt.sum(axis=0)
        tables.append(union.sum(axis=0) if saliency == 1 else union.T @ union - np.diag(union.sum(axis=0)))
        per_file[chrom] = (fname, x, cnt)
    exp = orc.normalize_expected(np.sum(tables, axis=0))
    score = (lambda c, n: orc.s1_scores_from_counts(c, n, exp)) if saliency == 1 else \
        (lambda c, n: orc.s2_scores_from_counts(c, n * (n - 1), exp))
    rows = []
    for chrom in orderChromosomes(list(per_file)):
        fname, x, cnt = per_file[chrom]
        sc = np.stack([score(cnt[g], n) for g, n in enumerate(sizes)]).astype(np.float32)
        t, g, s, sign = mgo.stat_and_driver(sc, sizes)
        k = (draw_exceedances(cnt, sizes, t, P, file_seed(seed, fname.split(".")[0]), 0, saliency, exp, score)
             if P else None)
        for r in range(len(t)):
            rows.append((chrom, r * 200, r * 200 + 200, t[r], g[r], s[r], sign[r], None if k is None else k[r]))
    t = np.array([r[3] for r in rows])
    pv = bh = None
    if P:
        k = np.array([r[7] for r in rows])
        pv = (1.0 + k) / (P + 1.0)
        bh = pso.bh(pv)
    metrics = ""
    for i, (chrom, st, en, tv, g, s, sg, kk) in enumerate(rows):
        metrics += "%s\t%d\t%d\t%.5e\t%s\t%s\t%s" % (chrom, st, en, tv, names[g], STATE_NAMES[s], "-" if sg < 0 else "+")
        metrics += ("\t%d\t%.5e\t%.5e\n" % (kk, pv[i], bh[i])) if P else "\n"
    starts = np.array([r[1] for r in rows]); ends = np.array([r[2] for r in rows])
    sel = max_mean(starts, ends, t, roi_width, 100)
    roi = ""
    half = roi_width // 2
    for i, idx in enumerate(sel["original_idx"]):
        lo, hi = max(idx - half, 0), idx + half + (1 if roi_width % 2 else 0)
        b = lo + int(np.argmax(t[lo:hi]))
        _, _, _, tv, g, s, sg, _ = rows[b]
        roi += "%s\t%d\t%d\t%s\t%s\t%s\t%.5e" % (rows[idx][0], sel["start"][i], sel["end"][i], names[g], STATE_NAMES[s],
                                                 "-" if sg < 0 else "+", tv)
        roi += ("\t%.5e\t%.5e\n" % (pv[b], bh[b])) if P else "\n"
    return metrics, roi, sizes


def read_gz(path):
    with gzip.open(path, "rt") as f:
        return f.read()


@pytest.mark.parametrize("saliency", [1, 2])
@pytest.mark.parametrize("groups,P", [(("g1", "g4"), 0), (("g1", "g4"), 5), (("g2", "g5", "g1"), 4),
                                      (("g1", "g2", "g3", "g4", "g5"), 0), (("g1", "g2", "g3", "g4", "g5"), 3)])
def test_metrics_and_regions_against_numpy(tmp_path, monkeypatch, saliency, groups, P):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "31")
    inp, gfile, meta, data = inputs(tmp_path)
    out = tmp_path / "out"
    extra = ["--null-permutations", P] if P else []
    ok(run_cli(monkeypatch, "-m", "paired", "-i", inp, "-o", out, "-j", meta, "--groups", gfile, "-s", saliency,
               "-w", 9, "--multigroup", ",".join(groups), *extra))
    d = out / "_".join(groups)
    tag = "%s_s%d" % ("_".join(groups), saliency)
    assert sorted(p.name for p in d.iterdir()) == sorted(["multigroupMetrics_%s.txt.gz" % tag,
                                                          "regionsOfInterest_%s.txt" % tag])
    metrics, roi, sizes = expected_outputs(data, {g: MCOLS[g] for g in groups}, saliency, P, 31, 9)
    assert read_gz(d / ("multigroupMetrics_%s.txt.gz" % tag)) == metrics
    assert (d / ("regionsOfInterest_%s.txt" % tag)).read_text() == roi


def test_all_quiescent_bins_have_t_zero_and_p_one(tmp_path, monkeypatch):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "5")
    inp, gfile, meta, data = inputs(tmp_path)
    out = tmp_path / "out"
    ok(run_cli(monkeypatch, "-m", "paired", "-i", inp, "-o", out, "-j", meta, "--groups", gfile, "-s", 1, "-w", 9,
               "--multigroup", "g1,g2,g3", "--null-permutations", 6))
    lines = read_gz(out / "g1_g2_g3" / "multigroupMetrics_g1_g2_g3_s1.txt.gz").splitlines()
    rows = []
    for fname, (chrom, x) in sorted(data.items()):
        rows += [(chrom, r) for r in range(len(x)) if np.all(x[r, :15] == x[r, 0])]
    assert rows
    by_loc = {(ln.split("\t")[0], int(ln.split("\t")[1]) // 200): ln.split("\t") for ln in lines}
    for chrom, r in rows:
        f = by_loc[(chrom, r)]
        assert float(f[3]) == 0.0 and f[7] == "6" and float(f[8]) == 1.0


def test_several_comparisons_in_one_run_equal_runs_alone(tmp_path, monkeypatch):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "9")
    from epilogos_b200 import helpers
    inp, gfile, meta, _ = inputs(tmp_path)
    common = ["-m", "paired", "-i", inp, "-j", meta, "--groups", gfile, "-s", 2, "-w", 9, "--null-permutations", 3]
    be = MultiBackend()
    parsed = []
    real_read = helpers.read_matrix
    monkeypatch.setattr(helpers, "read_matrix", lambda *a, **k: parsed.append(str(a[0])) or real_read(*a, **k))
    all_out = tmp_path / "all"
    ok(run_cli(monkeypatch, *common, "-o", all_out, "--multigroup", "g1,g2,g3", "--multigroup", "g4,g5",
               "--compare", "g1:g5", backend=be))
    assert be.calls["group_counts"] == 2 and len(parsed) == len(set(parsed)) == 2
    for args, name in ((["--multigroup", "g1,g2,g3"], "g1_g2_g3"), (["--multigroup", "g4,g5"], "g4_g5"),
                       (["--compare", "g1:g5"], "g1_vs_g5")):
        alone = tmp_path / ("alone_" + name)
        ok(run_cli(monkeypatch, *common, "-o", alone, *args))
        assert_same_outputs(all_out / name, alone / name)


def test_temp_files_equal_the_hand_over(tmp_path, monkeypatch):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "13")
    inp, gfile, meta, _ = inputs(tmp_path)
    common = ["-m", "paired", "-i", inp, "-j", meta, "--groups", gfile, "-s", 1, "-w", 9, "--multigroup", "g1,g3,g5",
              "--null-permutations", 4]
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "mem"))
    monkeypatch.setenv("EPILOGOS_B200_KEEP_TEMP", "1")
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "files"))
    assert_same_outputs(tmp_path / "files" / "g1_g3_g5", tmp_path / "mem" / "g1_g3_g5")


GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
os.environ["EPILOGOS_B200_SHARD"] = {shard!r}
os.environ["EPILOGOS_B200_SEED"] = "17"
import torch.distributed as td
from test_multigroup import MultiBackend
from epilogos_b200 import session, run
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
session._backend = MultiBackend()
run.main.main({args!r}, standalone_mode=False)
td.destroy_process_group()
"""


@pytest.mark.parametrize("shard", ["rows", "files"])
def test_two_gloo_ranks_equal_one(tmp_path, monkeypatch, shard):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "17")
    inp, _, meta, data = make_inputs(tmp_path, files=(("chr1", 130), ("chr2", 90), ("chr3", 70)))
    gfile = tmp_path / "mgroups.tsv"
    gfile.write_text(MGROUPS)
    args = ["-m", "paired", "-i", str(inp), "-j", str(meta), "-s", "1", "-w", "9", "--groups", str(gfile),
            "--multigroup", "g1,g2,g4", "--null-permutations", "3"]
    one = tmp_path / "one"
    ok(run_cli(monkeypatch, "-o", one, *args))
    two = tmp_path / "two"
    port = 37500 + (os.getpid() % 2000) + (7 if shard == "files" else 0)
    code = GLOO_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), shard=shard, port=port,
                              args=["-o", str(two)] + args)
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    assert_same_outputs(two / "g1_g2_g4", one / "g1_g2_g4")
