"""Biosample groups (`--groups`, epilogos_b200.groups) on CPU: the group file, the flag rules, and group runs of the
command line against runs on column-subset files, on a stand-in backend.  The kernels are covered by
test_groups_gpu.py."""
import gzip
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
from click.testing import CliRunner

from oracle import epilogos_oracle as orc
from test_cli import META
from test_host_stages import ROOT, write_tsv
from test_pairwise_stats import StatsBackend

K = 18
COLS = 24
GROUPS = """# name<TAB>columns (1-based)
a\t1-8
b\t9-24

c\t20,5-12
one\t7
all\t1-24
u\t17,3,11-13
"""
COLUMNS = {"a": range(0, 8), "b": range(8, 24), "c": list(range(4, 12)) + [19], "one": [6], "all": range(24),
           "u": [2, 10, 11, 12, 16]}


class GroupBackend(StatsBackend):
    """StatsBackend (an OracleBackend) plus the group entry points and S3, answered with numpy; counts its calls."""

    def __init__(self):
        self.calls = {"group_counts": 0, "gather_columns": 0}

    def states_to_device(self, states0):
        on_device = getattr(states0, "device_matrix", None)
        return on_device() if on_device is not None else torch.from_numpy(np.array(states0, dtype=np.int8))

    def gather_columns(self, x_dev, cols, idx):
        self.calls["gather_columns"] += 1
        assert x_dev.shape[1] == cols
        return torch.from_numpy(np.ascontiguousarray(x_dev.numpy()[:, np.asarray(idx)]))

    def group_counts(self, x_dev, cols, num_states, groups):
        self.calls["group_counts"] += 1
        x = x_dev.numpy()
        return torch.from_numpy(np.stack([orc.bin_counts(x[:, np.asarray(g)], num_states) for g in groups])
                                .astype(np.uint16).view(np.int16))

    def s3_tiles(self, x_dev, width, num_states):
        return torch.from_numpy(orc.s3_expected_counts(x_dev.numpy(), num_states).astype(np.int64)), {}

    def s3_counts(self, tiles, plan, width, num_states, total_bins):
        return tiles

    def scores_s3(self, x_dev, width, num_states, exp):
        return torch.from_numpy(orc.s3_scores_f64(x_dev.numpy(), num_states, exp.numpy()).astype(np.float32))


def make_matrix(rows=260, seed=1):
    rng = np.random.default_rng(seed)
    x = rng.integers(0, K, size=(rows, COLS), dtype=np.int8)
    x[rng.random(rows) < 0.2] = K - 1                                   # quiescent bins
    x[:40:3, :12] = rng.integers(0, 3, size=(len(range(0, 40, 3)), 12))   # some structure between the halves
    return x


def make_inputs(tmp_path, files=(("chr1", 260), ("chr2", 190))):
    inp = tmp_path / "in"
    inp.mkdir()
    data = {}
    for i, (chrom, rows) in enumerate(files):
        x = make_matrix(rows, seed=i + 1)
        name = "epilogos_matrix_%s.txt.gz" % chrom
        write_tsv(inp / name, x, chrom=chrom, gz=True)
        data[name] = (chrom, x)
    gfile = tmp_path / "groups.tsv"
    gfile.write_text(GROUPS)
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    return inp, gfile, meta, data


def subset_dir(tmp_path, data, name):
    """The directory of column-subset files of a group, named after it (what `cut -f` gives)."""
    d = tmp_path / "subsets" / name
    if not d.exists():
        d.mkdir(parents=True)
        for fname, (chrom, x) in data.items():
            write_tsv(d / fname, x[:, np.asarray(COLUMNS[name])], chrom=chrom, gz=True)
    return d


def cli(monkeypatch, backend, *args):
    from epilogos_b200 import run, session
    session.clear()
    monkeypatch.setattr(session, "_backend", backend)
    r = CliRunner().invoke(run.main, [str(a) for a in args])
    session.clear()
    assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)
    return r.output


def assert_same_outputs(got_dir, want_dir):
    got = sorted(p.name for p in Path(got_dir).iterdir())
    want = sorted(p.name for p in Path(want_dir).iterdir())
    assert got == want and got
    for name in got:
        a, b = Path(got_dir) / name, Path(want_dir) / name
        if name.endswith(".gz"):
            assert gzip.open(a).read() == gzip.open(b).read(), name
        elif name.endswith(".npy"):
            x, y = np.load(a), np.load(b)
            assert x.dtype == y.dtype and x.tobytes() == y.tobytes(), name
        elif name.endswith(".npz"):
            x, y = np.load(a, allow_pickle=True), np.load(b, allow_pickle=True)     # locations are object arrays
            assert sorted(x.files) == sorted(y.files)
            for k in x.files:
                same = np.array_equal(x[k], y[k]) if x[k].dtype == object else x[k].tobytes() == y[k].tobytes()
                assert x[k].dtype == y[k].dtype and same, (name, k)
        else:
            assert a.read_bytes() == b.read_bytes(), name


# ---- the group file ------------------------------------------------------------------------------------------------------

def test_group_file_parsing(tmp_path):
    from epilogos_b200 import groups
    f = tmp_path / "g.tsv"
    f.write_text(GROUPS)
    gs = groups.parseGroups(f)
    assert gs.names == ["a", "b", "c", "one", "all", "u"]
    for name, cols in COLUMNS.items():
        assert gs.columns[gs.index[name]].tolist() == sorted(cols)
    assert groups.parseComparisons(["a:b", "c:u"], gs) == [("a", "b"), ("c", "u")]
    with pytest.raises(ValueError, match="group 'b' uses biosample 24, but f.txt has 20 biosamples"):
        gs.check_width(20, "f.txt")


@pytest.mark.parametrize("text, message", [
    ("a 1-3\n", "line 1: expected 'name<TAB>columns'"),
    ("a\t1\tx\n", "line 1: expected 'name<TAB>columns'"),
    ("a\t1-x\n", "line 1: '1-x' is not a biosample number"),
    ("a\t0\n", "line 1: '0' is not a biosample number"),
    ("a\t5-3\n", "line 1: '5-3' is not a biosample number"),
    ("# c\n\na\t \n", "line 3: group 'a' has no columns"),
    ("a\t1,3,2-4\n", "line 1: group 'a' lists biosample 3 more than once"),
    ("a b\t1\n".replace(" ", "/"), "group name 'a/b' must match"),
    ("\t1\n", "group name '' must match"),
    ("a\t1\nb\t2\na\t3\n", "line 3: group name 'a' is used twice"),
    ("".join("g%d\t%d\n" % (i, i + 1) for i in range(65)), "more than 64 groups"),
    ("# nothing\n", "no group in"),
])
def test_group_file_errors(tmp_path, text, message):
    from epilogos_b200 import groups
    f = tmp_path / "g.tsv"
    f.write_text(text)
    with pytest.raises(groups.GroupFileError) as e:
        groups.parseGroups(f)
    assert str(e.value).startswith("ERROR: [--groups]") and message in str(e.value)


def test_sixty_four_groups_are_allowed(tmp_path):
    from epilogos_b200 import groups
    f = tmp_path / "g.tsv"
    f.write_text("".join("g%d\t%d\n" % (i, i + 1) for i in range(64)))
    assert len(groups.parseGroups(f)) == 64


def test_group_flag_rules(tmp_path):
    from epilogos_b200 import run
    g = tmp_path / "g.tsv"
    g.write_text(GROUPS)
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    inp = tmp_path / "in"
    inp.mkdir()
    (inp / "f.txt").write_text("chr1\t0\t200\t1\n")
    base = ["-o", str(tmp_path / "o"), "-j", str(meta)]
    cases = [
        (["--groups", g] + base, "ERROR: [--groups] requires [-i, --input-directory]"),
        (["-i", inp, "-a", inp, "--groups", g] + base, "ERROR: [--groups] not compatible with [-a, --directory-one]"),
        (["-i", inp, "-b", inp, "--groups", g] + base, "ERROR: [--groups] not compatible with [-b, --directory-two]"),
        (["-i", inp, "-f", "t", "--groups", g] + base, "ERROR: [--groups] not compatible with [-f, --file-tag]"),
        (["-i", inp, "--compare", "a:b"] + base, "ERROR: [--compare] requires [--groups]"),
        (["-i", inp, "--groups", g, "--compare", "a:b"] + base, "ERROR: [--compare] requires [-m, --mode] 'paired'"),
        (["-m", "paired", "-i", inp, "--groups", g] + base, "requires at least one [--compare]"),
        (["-m", "paired", "-i", inp, "--groups", g, "--compare", "a:x"] + base, "group 'x' is not defined"),
        (["-m", "paired", "-i", inp, "--groups", g, "--compare", "a:a"] + base, "compares a group with itself"),
        (["-m", "paired", "-i", inp, "--groups", g, "--compare", "ab"] + base, "is not of the form A:B"),
        (["-i", inp, "--groups", tmp_path / "missing.tsv"] + base, "ERROR: [--groups] cannot read"),
    ]
    for args, message in cases:
        r = CliRunner().invoke(run.main, [str(a) for a in args])
        assert message in r.output, (args, r.output)
        assert r.output.count("ERROR") == 1
        assert not (tmp_path / "o").exists()


def test_a_column_beyond_the_file_raises(tmp_path, monkeypatch):
    from epilogos_b200 import run, session
    inp, _, meta, _ = make_inputs(tmp_path, files=(("chr1", 50),))
    g = tmp_path / "wide.tsv"
    g.write_text("ok\t1-3\nwide\t2,25\n")
    session.clear()
    monkeypatch.setattr(session, "_backend", GroupBackend())
    r = CliRunner().invoke(run.main, ["-i", str(inp), "-o", str(tmp_path / "o"), "-j", str(meta), "--groups", str(g)])
    session.clear()
    assert isinstance(r.exception, ValueError)
    assert "group 'wide' uses biosample 25" in str(r.exception) and "epilogos_matrix_chr1.txt.gz" in str(r.exception)


# ---- single mode ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("saliency", [1, 2, 3])
def test_single_groups_equal_runs_on_subset_files(tmp_path, monkeypatch, saliency):
    from epilogos_b200 import helpers
    inp, gfile, meta, data = make_inputs(tmp_path)
    parsed = []
    real = helpers.read_matrix
    monkeypatch.setattr(helpers, "read_matrix", lambda *a, **k: (parsed.append(Path(a[0]).name), real(*a, **k))[1])
    be = GroupBackend()
    out = tmp_path / "out"
    log = cli(monkeypatch, be, "-i", inp, "-o", out, "-j", meta, "-s", saliency, "-w", 9, "--groups", gfile)
    assert "STEP 4" in log
    assert sorted(parsed) == sorted(data)                              # every file parsed once
    assert be.calls["group_counts"] == (len(data) if saliency != 3 else 0)
    assert be.calls["gather_columns"] == (len(data) * len(COLUMNS) if saliency == 3 else 0)
    assert sorted(p.name for p in out.iterdir()) == sorted(COLUMNS)
    for name in COLUMNS:
        want = tmp_path / "want" / name
        cli(monkeypatch, GroupBackend(), "-i", subset_dir(tmp_path, data, name), "-o", want, "-j", meta, "-s", saliency,
            "-w", 9)
        assert_same_outputs(out / name, want)
        assert (out / name / ("regionsOfInterest_%s_s%d.txt" % (name, saliency))).exists()


def test_single_groups_keep_temp_files_equal(tmp_path, monkeypatch):
    """With the in-memory hand-over off, the score stage writes the same temp files as the subset-file run."""
    monkeypatch.setenv("EPILOGOS_B200_KEEP_TEMP", "1")
    from epilogos_b200 import expected, expectedCombination, scores, session, groups
    inp, gfile, meta, data = make_inputs(tmp_path, files=(("chr1", 120),))
    gs = groups.parseGroups(gfile)
    f = next(inp.iterdir())
    be = GroupBackend()
    for name in ("c", "u"):
        got, want = tmp_path / "got" / name, tmp_path / "want" / name
        got.mkdir(parents=True); want.mkdir(parents=True)
        tag = "%s_s2" % name
        for d, src, sel in ((got, f, gs.select(name)), (want, subset_dir(tmp_path, data, name) / f.name, None)):
            session.clear()
            expected.main(src, "null", K, 2, d, tag, 1, False, backend=be, group=sel)
            expectedCombination.main(d, d / ("exp_freq_%s.npy" % tag), tag, False, backend=be)
            scores.main(src, "null", K, 2, d, d / ("exp_freq_%s.npy" % tag), tag, 1, K - 1, -1, False, backend=be,
                        group=sel)
        assert_same_outputs(got, want)
    session.clear()


# ---- paired mode ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("null_mode, extra", [("device", []), ("device", ["-g", "6", "-q", "0"]), ("reference", []),
                                              ("reference", ["-g", "6", "-q", "0"])])
def test_paired_groups_equal_two_directory_runs(tmp_path, monkeypatch, null_mode, extra):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "23")
    monkeypatch.setenv("EPILOGOS_B200_NULL", null_mode)
    from epilogos_b200 import helpers
    inp, gfile, meta, data = make_inputs(tmp_path)
    # the replay null draws from numpy's global generator, in file order: one comparison per run keeps the draws aligned
    comparisons = [("a", "b"), ("c", "u")] if null_mode == "device" else [("c", "u")]
    parsed = []
    real = helpers.read_matrix
    monkeypatch.setattr(helpers, "read_matrix", lambda *a, **k: (parsed.append(Path(a[0]).name), real(*a, **k))[1])
    be = GroupBackend()
    out = tmp_path / "out"
    common = ["-j", meta, "-s", 1 if extra else 2, "-w", 9, "-n", "-t", 3, "-z", 150] + extra
    np.random.seed(4)
    cli(monkeypatch, be, "-m", "paired", "-i", inp, "-o", out, "--groups", gfile,
        *sum((["--compare", "%s:%s" % c] for c in comparisons), []), *common)
    assert sorted(parsed) == sorted(data) and be.calls["group_counts"] == len(data)
    monkeypatch.setattr(helpers, "read_matrix", real)
    for a, b in comparisons:
        got = out / ("%s_vs_%s" % (a, b))
        want = tmp_path / "want" / got.name
        np.random.seed(4)
        cli(monkeypatch, GroupBackend(), "-m", "paired", "-a", subset_dir(tmp_path, data, a), "-b",
            subset_dir(tmp_path, data, b), "-o", want, *common)
        assert_same_outputs(got, want)
        tag = "%s_%s_s%d" % (a, b, 1 if extra else 2)
        assert (got / ("pairwiseMetrics_%s.txt.gz" % tag)).exists() and (got / ("regionsOfInterest_%s.txt" % tag)).exists()


# ---- several ranks -------------------------------------------------------------------------------------------------------

GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
os.environ["EPILOGOS_B200_SHARD"] = {shard!r}
import torch.distributed as td
from test_groups import GroupBackend
from epilogos_b200 import session, run
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
session._backend = GroupBackend()
run.main.main({args!r}, standalone_mode=False)
td.destroy_process_group()
"""


@pytest.mark.parametrize("shard", ["rows", "files"])
def test_two_gloo_ranks_write_the_same_group_outputs_as_one(tmp_path, monkeypatch, shard):
    inp, gfile, meta, data = make_inputs(tmp_path, files=(("chr1", 230), ("chr2", 150), ("chr3", 90)))
    args = ["-i", str(inp), "-j", str(meta), "-s", "2", "-w", "9", "--groups", str(gfile)]
    one = tmp_path / "one"
    cli(monkeypatch, GroupBackend(), "-o", one, *args)
    two = tmp_path / "two"
    port = 36500 + (os.getpid() % 2000) + (7 if shard == "files" else 0)
    code = GLOO_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), shard=shard, port=port,
                              args=["-o", str(two)] + args)
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    for name in COLUMNS:
        assert_same_outputs(two / name, one / name)
