"""Stratified permutations (--strata) on a stand-in backend: the flag and load-time rules with their messages and
precedence, the column numbering, byte-identity of every output with one stratum holding every biosample, the outputs
with several strata against numpy (tests/strata_oracle.py), the stratified region splits, and gloo ranks in both
sharding modes.  The kernels are covered by test_strata_gpu.py."""
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from click.testing import CliRunner

import multigroup_oracle as mgo
import region_oracle as ro
import strata_oracle as sto
from oracle import epilogos_oracle as orc
from test_groups import K, assert_same_outputs, make_inputs
from test_host_stages import ROOT
from test_multigroup import MGROUPS
from test_pairwise_stats import make_paired_inputs
from test_region_permutations import RegionBackend

W = 9
AB_STRATA = "t1\t1-10,31-45\nt2\t11-25,46-50\nonlyA\t26-30\nonlyB\t51-55\n"      # over [A | B] = 30 + 25 columns
AB_ALL = "all\t1-55\n"
I_STRATA = "s1\t1-6,13-18\ns2\t7-12,19-24\n"                                    # over the 24 columns of -i
I_ALL = "everything\t1-24\n"


class StrataBackend(RegionBackend):
    """The stand-in plus the stratified routes, answered by strata_oracle; without strata every method is the parent's."""

    def stratum_counts(self, x_dev, cols, num_states, columns):
        return torch.from_numpy(sto.stratum_counts(np.asarray(x_dev)[:, :cols], columns, num_states)
                                .astype(np.uint16).view(np.int16))

    def _draw(self, strata, seed, nperm, bin_offset):
        return sto.shuffled_counts(self._cnt(strata.counts), strata.sizes, seed, nperm, bin_offset)

    def shuffled_counts_device(self, cnt_a, cnt_b, size_a, size_b, seed, nperm=1, width=None, bin_offset=0, strata=None):
        if strata is None:
            return super().shuffled_counts_device(cnt_a, cnt_b, size_a, size_b, seed, nperm, width, bin_offset)
        t = torch.from_numpy(self._draw(strata, seed, nperm, bin_offset).astype(np.uint16).view(np.int16))
        return (t[0, 0], t[0, 1]) if nperm == 1 else (t[:, 0], t[:, 1])

    def permutation_exceedances(self, cnt_a, cnt_b, dist, nperm, seed, size_a, size_b, width, bin_offset, saliency, exp,
                                score_widths, perms, exact=False, workspace_bytes=None, strata=None):
        if strata is None:
            return super().permutation_exceedances(cnt_a, cnt_b, dist, nperm, seed, size_a, size_b, width, bin_offset,
                                                   saliency, exp, score_widths, perms, exact)
        x = self._draw(strata, seed, nperm, bin_offset)
        rows, k = cnt_a.shape
        flat = [torch.from_numpy(x[:, g].reshape(-1, k).astype(np.uint16).view(np.int16)) for g in range(2)]
        sa = self.scores(flat[0], score_widths[0], saliency, exp, perms=perms[0])
        sb = self.scores(flat[1], score_widths[1], saliency, exp, perms=perms[1])
        _, null = self.pairwise_combine(None, None, sa, sb)
        null = null.numpy().astype(np.float32).reshape(nperm, rows)
        counts = (np.abs(null) >= np.abs(np.asarray(dist, dtype=np.float32))).sum(axis=0).astype(np.uint32)
        return torch.from_numpy(counts.view(np.int32))

    def multigroup_exceedances(self, cnt, sizes, t, nperm, seed, bin_offset, saliency, exp, exact=False,
                               workspace_bytes=None, strata=None):
        if strata is None:
            return super().multigroup_exceedances(cnt, sizes, t, nperm, seed, bin_offset, saliency, exp)
        x = self._draw(strata, seed, nperm, bin_offset)
        score = self._score_fn(saliency, exp)
        null = np.stack([np.stack([score(x[p, g], n) for g, n in enumerate(sizes)]) for p in range(nperm)])
        k = mgo.exceedances(null.astype(np.float32), sizes, t.numpy())
        return torch.from_numpy(k.astype(np.uint32).view(np.int32))

    def _strata_maxima(self, x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, stat, strata):
        x = np.asarray(x_dev)[:, :sum(sizes)]
        if halo is not None and len(halo):
            x = np.concatenate([x, np.asarray(halo)])
        e = np.asarray(exp)
        return torch.from_numpy(sto.file_maxima(x, num_states, strata.positions, strata.sizes, window, nperm, seed,
                                                lambda cnt: stat(cnt, sizes, saliency, e)))

    def region_maxima_paired(self, x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, exact=False,
                             strata=None):
        if strata is None:
            return super().region_maxima_paired(x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp)
        return self._strata_maxima(x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, ro.paired_stat,
                                   strata)

    def region_maxima_multigroup(self, x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, exact=False,
                                 strata=None):
        if strata is None:
            return super().region_maxima_multigroup(x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp)
        return self._strata_maxima(x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp,
                                   ro.multigroup_stat, strata)


def run_cli(monkeypatch, *args, backend=None):
    from epilogos_b200 import run, session
    session.clear()
    monkeypatch.setattr(session, "_backend", backend or StrataBackend())
    r = CliRunner().invoke(run.main, [str(a) for a in args])
    session.clear()
    return r


def ok(r):
    assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)
    return r


def strata_file(tmp_path, text, name="strata.tsv"):
    f = tmp_path / name
    f.write_text(text)
    return f


def read_gz(path):
    with gzip.open(path, "rt") as f:
        return f.read()


# ---- the rules ----------------------------------------------------------------------------------------------------------

def test_flag_and_file_rules_and_their_precedence(tmp_path, monkeypatch, golden):
    a, b, meta = make_paired_inputs(tmp_path, golden)
    out = tmp_path / "out"
    good = strata_file(tmp_path, AB_STRATA)
    pab = ["-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta]
    bad = {name: strata_file(tmp_path, text, name + ".tsv") for name, text in [
        ("line", "t1 1-3\n"), ("name", "t/1\t1-3\n"), ("twice", "t1\t1-3\nt1\t4-5\n"), ("col", "t1\t1-3,2\n"),
        ("empty", "t1\t\n"), ("many", "".join("t%d\t%d\n" % (i, i + 1) for i in range(65))),
        ("share", "t1\t1-3\nt2\t4-6\nt3\t6-9\n")]}
    cases = [
        (["-i", a, "-o", out, "-j", meta, "--strata", good], "ERROR: [--strata] requires [-m, --mode] 'paired'"),
        (pab + ["-g", 10, "--strata", good], "ERROR: [--strata] not compatible with [-g, --group-size] option"),
        (pab + ["--strata", bad["line"]], "ERROR: [--strata] line 1: expected 'name<TAB>columns', got 't1 1-3'"),
        (pab + ["--strata", bad["name"]], "ERROR: [--strata] line 1: group name 't/1' must match [A-Za-z0-9._-]+"),
        (pab + ["--strata", bad["twice"]], "ERROR: [--strata] line 2: group name 't1' is used twice"),
        (pab + ["--strata", bad["col"]], "ERROR: [--strata] line 1: group 't1' lists biosample 2 more than once"),
        (pab + ["--strata", bad["empty"]], "ERROR: [--strata] line 1: group 't1' has no columns"),
        (pab + ["--strata", bad["many"]], "ERROR: [--strata] more than 64 groups in %s" % bad["many"]),
        (pab + ["--strata", bad["share"]], "ERROR: [--strata] strata 't2' and 't3' share biosample 6"),
        # the order among the new rules
        (["-i", a, "-o", out, "-j", meta, "-g", 10, "--strata", bad["line"]],
         "ERROR: [--strata] requires [-m, --mode] 'paired'"),
        (pab + ["-g", 10, "--strata", bad["line"]], "ERROR: [--strata] not compatible with [-g, --group-size] option"),
        # after every existing rule
        (pab + ["--strata", bad["line"], "--roi-permutations", 0],
         "ERROR: Number of region permutations must be between 1 and 100000"),
        (pab + ["--strata", bad["line"], "--null-permutations", 0],
         "ERROR: Number of null permutations must be between 1 and 1000000"),
        (pab + ["-g", 10, "--strata", good, "--roi-permutations", 3],
         "ERROR: [--roi-permutations] not compatible with [-g, --group-size] option"),
        (["-m", "paired", "-a", a, "-o", out, "-j", meta, "--strata", bad["line"]],
         "ERROR: [-b, --directory-two] required in 'paired' group mode"),
    ]
    for args, message in cases:
        r = run_cli(monkeypatch, *args)
        assert r.output.strip().splitlines()[-1] == message, (args, r.output)
        assert not list(out.glob("pairwise*"))
    r = run_cli(monkeypatch, *pab, "--strata", tmp_path / "missing.tsv")
    assert r.output.strip().splitlines()[-1].startswith("ERROR: [--strata] cannot read %s" % (tmp_path / "missing.tsv"))


def test_group_file_messages_are_unchanged(tmp_path):
    from epilogos_b200 import groups
    f = strata_file(tmp_path, "t1\t1-3,2\n")
    with pytest.raises(groups.GroupFileError) as e:
        groups.parseGroups(f)
    assert str(e.value) == "ERROR: [--groups] line 1: group 't1' lists biosample 2 more than once"


@pytest.mark.parametrize("text,env,match", [
    ("t1\t1-30\nt2\t31-56\n", None, r"stratum 't2' uses biosample 56, but .* has 55 biosamples"),
    ("t1\t1-30\nt2\t31-54\n", None, r"biosample 55 of the comparison \[-a\] vs \[-b\] is in no stratum"),
    ("t1\t1-30\nt2\t31-55\n", None, r"no stratum holds biosamples of two groups of the comparison \[-a\] vs \[-b\]"),
    (AB_STRATA, "reference", r"EPILOGOS_B200_NULL=reference"),
])
def test_load_time_rules_raise_naming_the_file(tmp_path, monkeypatch, golden, text, env, match):
    if env:
        monkeypatch.setenv("EPILOGOS_B200_NULL", env)
    a, b, meta = make_paired_inputs(tmp_path, golden)
    f = strata_file(tmp_path, text)
    r = run_cli(monkeypatch, "-m", "paired", "-a", a, "-b", b, "-o", tmp_path / "o", "-j", meta, "--strata", f)
    assert isinstance(r.exception, ValueError), r.output
    assert str(f) in str(r.exception)
    import re
    assert re.search(match, str(r.exception)), str(r.exception)


def test_the_header_names_the_strata(tmp_path, monkeypatch, golden):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "3")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    r = ok(run_cli(monkeypatch, "-m", "paired", "-a", a, "-b", b, "-o", tmp_path / "o", "-j", meta, "-w", W,
                   "--strata", strata_file(tmp_path, AB_STRATA)))
    assert "        Strata = 4 (biosamples per stratum: 25, 20, 5, 5)" in r.output.splitlines()


# ---- the numbering ------------------------------------------------------------------------------------------------------

def test_numbering_over_a_and_b_and_over_the_group_file(tmp_path):
    from epilogos_b200 import groups
    st = groups.parseStrata(strata_file(tmp_path, AB_STRATA))
    lay = st.layout([np.arange(30), 30 + np.arange(25)], "x", 55, "f")
    assert lay.names == ["t1", "t2", "onlyA", "onlyB"]
    assert lay.sizes == [[10, 15], [15, 5], [5, 0], [0, 5]]
    assert lay.positions[0].tolist() == list(range(10)) + list(range(30, 45))
    assert lay.columns[3].tolist() == list(range(50, 55))
    # --compare a:c, which share biosamples 5-8: they count in both groups, in their stratum
    st = groups.parseStrata(strata_file(tmp_path, I_STRATA + "unused\t25\n"))
    a, c = np.arange(0, 8), np.array(list(range(4, 12)) + [19])
    lay = st.layout([a, c], "a:c", 25, "f")
    assert lay.names == ["s1", "s2"] and lay.sizes == [[6, 2], [2, 7]]
    assert sorted(lay.columns[0].tolist()) == [0, 1, 2, 3, 4, 4, 5, 5]
    assert lay.positions[0].tolist() == [0, 1, 2, 3, 4, 5, 8, 9]
    assert lay.positions[1].tolist() == [6, 7, 10, 11, 12, 13, 14, 15, 16]


# ---- one stratum holding everything: every output as without --strata -----------------------------------------------------

@pytest.mark.parametrize("saliency", [1, 2])
@pytest.mark.parametrize("extra", [["-n", "-t", "3", "-z", "150"], ["--null-permutations", "5", "--roi-permutations", "4"]])
def test_one_stratum_is_byte_identical_two_directories(tmp_path, monkeypatch, golden, saliency, extra):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "5")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    common = ["-m", "paired", "-a", a, "-b", b, "-j", meta, "-s", saliency, "-w", W, *extra]
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "plain"))
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "strata", "--strata", strata_file(tmp_path, AB_ALL)))
    assert_same_outputs(tmp_path / "strata", tmp_path / "plain")


@pytest.mark.parametrize("saliency", [1, 2])
@pytest.mark.parametrize("what", [["--compare", "a:c"], ["--multigroup", "g2,g5,g1"],
                                  ["--multigroup", "g1,g2,g3,g4,g5"]])
def test_one_stratum_is_byte_identical_with_groups(tmp_path, monkeypatch, saliency, what):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "8")
    inp, _, meta, _ = make_inputs(tmp_path)
    gfile = strata_file(tmp_path, MGROUPS + "c\t20,5-12\n", "groups.tsv")
    common = ["-m", "paired", "-i", inp, "-j", meta, "--groups", gfile, "-s", saliency, "-w", W, *what,
              "--null-permutations", 4, "--roi-permutations", 3]
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "plain"))
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "strata", "--strata", strata_file(tmp_path, I_ALL)))
    d = what[1].replace(":", "_vs_").replace(",", "_")
    assert_same_outputs(tmp_path / "strata" / d, tmp_path / "plain" / d)


# ---- several strata against numpy ---------------------------------------------------------------------------------------

def ab_expectations(golden, P, R, run_seed, saliency=1):
    """(k per bin per file, region maxima) of the -a/-b run with AB_STRATA, from numpy."""
    from epilogos_b200 import groups
    from epilogos_b200.pairwise import file_seed
    g = golden("paired_synth_c30_c25_k18")
    x = np.concatenate([g["xa"], g["xb"]], axis=1).astype(np.int64)
    parts = np.array_split(np.arange(len(x)), 2)
    lay = groups.Strata(groups.GroupSet(
        ["t1", "t2", "onlyA", "onlyB"], [np.r_[0:10, 30:45], np.r_[10:25, 45:50], np.r_[25:30], np.r_[50:55]]),
        "f").layout([np.arange(30), 30 + np.arange(25)], "x", 55, "f")
    tables = []
    for rows in parts:
        u = orc.bin_counts(x[rows], K).astype(np.int64)
        tables.append(u.sum(axis=0) if saliency == 1 else u.T @ u - np.diag(u.sum(axis=0)))
    exp = orc.normalize_expected(np.sum(tables, axis=0))
    score = ro.score_fn(saliency, exp)
    ks, maxima = [], []
    for i, rows in enumerate(parts):
        xf = x[rows]
        ca, cb = orc.bin_counts(xf[:, :30], K).astype(np.int64), orc.bin_counts(xf[:, 30:], K).astype(np.int64)
        delta = np.asarray(score(ca, 30), dtype=np.float32) - np.asarray(score(cb, 25), dtype=np.float32)
        dist, _ = orc.paired_real_reductions(delta, round_trip=True)
        cnt_h = sto.stratum_counts(xf, lay.columns, K)
        d = sto.shuffled_counts(cnt_h, lay.sizes, file_seed(run_seed, "epilogos_matrix_chr%d" % (i + 1)), P)
        null = []
        for p in range(P):
            nd = np.asarray(score(d[p, 0], 30), dtype=np.float32) - np.asarray(score(d[p, 1], 25), dtype=np.float32)
            null.append(np.sum(np.square(nd), axis=1) * np.sign(np.sum(nd, axis=1)))
        null = np.array(null, dtype=np.float32)
        ks.append((np.abs(null) >= np.abs(np.asarray(dist, dtype=np.float32))).sum(axis=0))
        seed = file_seed(run_seed, ro.SEED_SALT)
        maxima.append(sto.file_maxima(xf, K, lay.positions, lay.sizes, W, R, seed,
                                      lambda cnt: ro.paired_stat(cnt, (30, 25), saliency, exp)))
    return np.concatenate(ks), np.max(maxima, axis=0), lay


@pytest.mark.parametrize("saliency", [1, 2])
def test_several_strata_against_numpy_two_directories(tmp_path, monkeypatch, golden, saliency):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "21")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    out = tmp_path / "out"
    ok(run_cli(monkeypatch, "-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta, "-s", saliency, "-w", W,
               "--null-permutations", 6, "--roi-permutations", 5, "--strata", strata_file(tmp_path, AB_STRATA)))
    k, maxima, _ = ab_expectations(golden, 6, 5, 21, saliency)
    tag = "a_b_s%d" % saliency
    got_k = [int(l.split("\t")[3]) for l in read_gz(out / ("pairwisePermutation_%s.txt.gz" % tag)).splitlines()]
    assert got_k == k.tolist()
    assert 0 < k.sum() < 6 * len(k)
    z = np.load(out / ("regionNullMaxima_%s.npz" % tag))
    assert z["maxima"].tolist() == maxima.tolist()
    # the plain outputs do not depend on the strata
    ok(run_cli(monkeypatch, "-m", "paired", "-a", a, "-b", b, "-o", tmp_path / "plain", "-j", meta, "-s", saliency,
               "-w", W))
    plain = sorted(f.name for f in (tmp_path / "plain").iterdir())
    assert plain and all((out / n).exists() for n in plain)
    for name in plain:
        a_, b_ = out / name, tmp_path / "plain" / name
        assert (read_gz(a_) == read_gz(b_)) if name.endswith(".gz") else a_.read_bytes() == b_.read_bytes(), name


def test_the_run_null_is_permutation_zero_of_the_strata(tmp_path, monkeypatch, golden):
    """The null that -n fits (temp_nullDistances, written by the score stage run on its own) is the stratified draw of
    permutation 0."""
    from epilogos_b200 import expected, expectedCombination, groups, scores, session
    from epilogos_b200.pairwise import file_seed
    monkeypatch.setenv("EPILOGOS_B200_SEED", "9")
    a, b, meta = make_paired_inputs(tmp_path, golden, chroms=("chr1",))
    out = tmp_path / "out"
    out.mkdir()
    be = StrataBackend()
    session.clear()
    fa, fb = a / "epilogos_matrix_chr1.txt.gz", b / "epilogos_matrix_chr1.txt.gz"
    expected.main(fa, fb, K, 1, out, "t", 1, False, backend=be)
    expectedCombination.main(out, out / "exp_freq_t.npy", "t", False, backend=be)
    scores.main(fa, fb, K, 1, out, out / "exp_freq_t.npy", "t", 1, K - 1, -1, False, backend=be,
                strata=groups.parseStrata(strata_file(tmp_path, AB_STRATA)))
    session.clear()
    null = np.load(out / "temp_nullDistances_t_epilogos_matrix_chr1.npz")["nullDistances"]
    g = golden("paired_synth_c30_c25_k18")
    x = np.concatenate([g["xa"], g["xb"]], axis=1).astype(np.int64)
    _, _, lay = ab_expectations(golden, 1, 1, 9)
    exp = np.load(out / "exp_freq_t.npy")
    d = sto.shuffled_counts(sto.stratum_counts(x, lay.columns, K), lay.sizes, file_seed(9, "epilogos_matrix_chr1"), 1)[0]
    nd = orc.s1_scores_from_counts(d[0], 30, exp) - orc.s1_scores_from_counts(d[1], 25, exp)
    want = (np.sum(np.square(nd), axis=1) * np.sign(np.sum(nd, axis=1))).astype(np.float32)
    assert null.tobytes() == want.tobytes()
    # every shuffle keeps the strata's make-up: A' gets 30 labels, those of stratum onlyA among them
    assert np.array_equal(d[0].sum(axis=1), np.full(len(x), 30))
    only_a = orc.bin_counts(x[:, 25:30], K)
    assert np.all(d[0] >= only_a)


def test_several_strata_multigroup_against_numpy(tmp_path, monkeypatch):
    from epilogos_b200.pairwise import file_seed
    monkeypatch.setenv("EPILOGOS_B200_SEED", "31")
    inp, _, meta, data = make_inputs(tmp_path)
    gfile = strata_file(tmp_path, MGROUPS, "groups.tsv")
    out = tmp_path / "out"
    groups_ = ("g2", "g5", "g1")
    ok(run_cli(monkeypatch, "-m", "paired", "-i", inp, "-o", out, "-j", meta, "--groups", gfile, "-w", W,
               "--multigroup", ",".join(groups_), "--null-permutations", 5, "--strata", strata_file(tmp_path, I_STRATA)))
    cols = [np.r_[5:10], np.r_[20:24], np.r_[0:5]]
    sizes = [len(c) for c in cols]
    s_of = np.array([0] * 6 + [1] * 6 + [0] * 6 + [1] * 6)
    st_sizes = [[int(np.sum(s_of[c] == h)) for c in cols] for h in (0, 1)]
    st_cols = [np.concatenate([c[s_of[c] == h] for c in cols]) for h in (0, 1)]
    tables, per = [], {}
    for fname, (chrom, x) in data.items():
        cnt = np.stack([orc.bin_counts(x[:, c], K) for c in cols]).astype(np.int64)
        tables.append(cnt.sum(axis=0).sum(axis=0))
        per[chrom] = (fname, x, cnt)
    exp = orc.normalize_expected(np.sum(tables, axis=0))
    score = ro.score_fn(1, exp)
    want = []
    for chrom in ("chr1", "chr2"):
        fname, x, cnt = per[chrom]
        t = mgo.statistic(np.stack([score(cnt[g], n) for g, n in enumerate(sizes)]).astype(np.float32), sizes)[0]
        d = sto.shuffled_counts(sto.stratum_counts(x, st_cols, K), st_sizes, file_seed(31, fname.split(".")[0]), 5)
        null = np.stack([np.stack([score(d[p, g], n) for g, n in enumerate(sizes)]) for p in range(5)])
        want += mgo.exceedances(null.astype(np.float32), sizes, t).tolist()
    name = "_".join(groups_)
    got = [int(l.split("\t")[7]) for l in read_gz(out / name / ("multigroupMetrics_%s_s1.txt.gz" % name)).splitlines()]
    assert got == want


# ---- the region splits ----------------------------------------------------------------------------------------------------

def test_region_splits_keep_each_groups_make_up_and_the_identity_is_the_real_split():
    from epilogos_b200 import region_null
    positions = [np.array([0, 1, 2, 7, 8]), np.array([3, 4, 9, 10, 11, 12]), np.array([5, 6])]
    sizes = [[3, 2], [2, 4], [2, 0]]
    N = 13
    stratum = np.zeros(N, dtype=int)
    for h, p in enumerate(positions):
        stratum[p] = h
    seen = set()
    for p0, members in region_null.split_blocks(5, (7, 6), 40, 7, strata=(positions, sizes)):
        for m in members:
            g0 = np.flatnonzero(np.unpackbits(m.view(np.uint8), bitorder="little")[:N])
            assert [int(np.sum(stratum[g0] == h)) for h in range(3)] == [3, 2, 2]
            seen.add(tuple(g0))
    assert len(seen) > 20
    # the same permutations as the oracle's
    want = [tuple(sorted(parts[0])) for parts in sto.splits(5, positions, sizes, 40)]
    got = []
    for _, members in region_null.split_blocks(5, (7, 6), 40, 3, strata=(positions, sizes)):
        got += [tuple(np.flatnonzero(np.unpackbits(m.view(np.uint8), bitorder="little")[:N])) for m in members]
    assert got == want
    # identity: each stratum's first n[h][0] positions are group 0's own columns
    ident = np.concatenate([p[:n[0]] for p, n in zip(positions, sizes)])
    assert sorted(ident.tolist()) == list(range(7))


# ---- several ranks -----------------------------------------------------------------------------------------------------

GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
os.environ["EPILOGOS_B200_SHARD"] = {shard!r}
os.environ["EPILOGOS_B200_SEED"] = "17"
import torch.distributed as td
from test_strata import StrataBackend
from epilogos_b200 import session, run
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
session._backend = StrataBackend()
run.main.main({args!r}, standalone_mode=False)
td.destroy_process_group()
"""


@pytest.mark.parametrize("shard", ["rows", "files"])
def test_two_gloo_ranks_equal_one(tmp_path, monkeypatch, shard):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "17")
    inp, _, meta, _ = make_inputs(tmp_path, files=(("chr1", 130), ("chr2", 70)))
    gfile = strata_file(tmp_path, MGROUPS + "c\t20,5-12\n", "groups.tsv")
    args = ["-m", "paired", "-i", str(inp), "-j", str(meta), "-s", "1", "-w", "20", "--groups", str(gfile),
            "--multigroup", "g1,g2,g4", "--compare", "a:c", "--null-permutations", "4", "--roi-permutations", "3",
            "--strata", str(strata_file(tmp_path, I_STRATA))]
    one = tmp_path / "one"
    ok(run_cli(monkeypatch, "-o", one, *args))
    many = tmp_path / "many"
    port = 40100 + (os.getpid() % 1500) + (7 if shard == "files" else 0)
    code = GLOO_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), shard=shard, port=port,
                              args=["-o", str(many)] + args)
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    for d in ("g1_g2_g4", "a_vs_c"):
        assert_same_outputs(many / d, one / d)
