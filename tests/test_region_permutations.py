"""Family-wise p-values of the regions of interest (--roi-permutations P) on a stand-in backend: the flag rules, both output
files against the numpy oracle (tests/region_oracle.py) for -a/-b, --compare and --multigroup, byte-identity of every other
output, the temp-file route, gloo ranks in both sharding modes, one seed per run, and the one-chromosome rule.  The kernels
are covered by test_region_permutations_gpu.py."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from click.testing import CliRunner

import region_oracle as ro
from oracle import epilogos_oracle as orc
from test_groups import COLUMNS, K, assert_same_outputs, make_inputs
from test_host_stages import ROOT
from test_multigroup import MCOLS, MGROUPS, MultiBackend
from test_pairwise_stats import make_paired_inputs

W = 9


class RegionBackend(MultiBackend):
    """The stand-in plus the region null, answered by the numpy oracle on the rows it is given (own rows + halo)."""

    def _maxima(self, x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, stat):
        x = np.asarray(x_dev)[:, :sum(sizes)]
        if halo is not None and len(halo):
            x = np.concatenate([x, np.asarray(halo)])
        e = np.asarray(exp)
        return torch.from_numpy(ro.file_maxima(x, num_states, sizes, window, nperm, seed,
                                               lambda cnt: stat(cnt, sizes, saliency, e)))

    def region_maxima_paired(self, x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, exact=False):
        return self._maxima(x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, ro.paired_stat)

    def region_maxima_multigroup(self, x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, exact=False):
        return self._maxima(x_dev, halo, sizes, num_states, window, nperm, seed, saliency, exp, ro.multigroup_stat)


def run_cli(monkeypatch, *args, backend=None):
    from epilogos_b200 import run, session
    session.clear()
    monkeypatch.setattr(session, "_backend", backend or RegionBackend())
    r = CliRunner().invoke(run.main, [str(a) for a in args])
    session.clear()
    return r


def ok(r):
    assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)


def region_seed(run_seed):
    from epilogos_b200.pairwise import file_seed
    return file_seed(run_seed, ro.SEED_SALT)


def expected(files, sizes, saliency, P, run_seed, kind):
    """(regionPermutation text, maxima) from numpy: files = {chrom: x [rows, N]} with the groups as consecutive column
    slices of `sizes`."""
    from epilogos_b200.roi import orderChromosomes
    tables = []
    for x in files.values():
        union = orc.bin_counts(x, K).astype(np.int64)
        tables.append(union.sum(axis=0) if saliency == 1 else union.T @ union - np.diag(union.sum(axis=0)))
    exp = orc.normalize_expected(np.sum(tables, axis=0))
    stat = ro.paired_stat if kind == "paired" else ro.multigroup_stat
    seed = region_seed(run_seed)
    order = orderChromosomes(list(files))
    maxima = np.max([ro.file_maxima(files[c], K, sizes, W, P, seed, lambda cnt: stat(cnt, sizes, saliency, exp))
                     for c in order], axis=0)
    xs, chrom, starts = [], [], []
    for c in order:
        x = files[c]
        ident = ro.group_counts(x, K, np.arange(x.shape[1]), sizes)
        xs.append(stat(ident, sizes, saliency, exp))
        chrom += [c] * len(x)
        starts.append(np.arange(len(x)) * 200)
    starts = np.concatenate(starts)
    xv = np.concatenate(xs)
    return ro.region_text(np.array(chrom, dtype=object), starts, starts + 200, xv, W, maxima), maxima


def check_outputs(d, tag, text, maxima, P):
    assert (d / ("regionPermutation_%s.txt" % tag)).read_text() == text
    z = np.load(d / ("regionNullMaxima_%s.npz" % tag))
    assert z["maxima"].dtype == np.int64 and z["maxima"].tolist() == maxima.tolist()
    assert int(z["window"]) == W and int(z["permutations"]) == P
    assert not list(d.glob("temp_*"))


def strip_region_files(d, tag):
    for name in ("regionPermutation_%s.txt" % tag, "regionNullMaxima_%s.npz" % tag):
        (d / name).unlink()


# ---- the flag rules ---------------------------------------------------------------------------------------------------

def test_flag_rules_and_their_precedence(tmp_path, monkeypatch, golden):
    a, b, meta = make_paired_inputs(tmp_path, golden)
    out = tmp_path / "out"
    pab = ["-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta]
    cases = [
        (["-i", a, "-o", out, "-j", meta, "--roi-permutations", 5],
         "ERROR: [--roi-permutations] requires [-m, --mode] 'paired'"),
        (pab + ["--roi-permutations", 0], "ERROR: Number of region permutations must be between 1 and 100000"),
        (pab + ["--roi-permutations", 100001], "ERROR: Number of region permutations must be between 1 and 100000"),
        (pab + ["--roi-permutations", 5, "-g", 10], "ERROR: [--roi-permutations] not compatible with [-g, --group-size] option"),
        (pab + ["--roi-permutations", 5, "-w", 16385],
         "ERROR: [--roi-permutations] needs a region width [-w, --roi-width] of at most 16384 bins"),
        # the order among the new rules
        (["-i", a, "-o", out, "-j", meta, "--roi-permutations", 0, "-g", 10],
         "ERROR: [--roi-permutations] requires [-m, --mode] 'paired'"),
        (pab + ["--roi-permutations", 0, "-g", 10], "ERROR: Number of region permutations must be between 1 and 100000"),
        (pab + ["--roi-permutations", 5, "-g", 10, "-w", 20000],
         "ERROR: [--roi-permutations] not compatible with [-g, --group-size] option"),
        # after every existing rule
        (pab + ["--roi-permutations", 0, "--null-permutations", 0],
         "ERROR: Number of null permutations must be between 1 and 1000000"),
        (pab + ["--roi-permutations", 0, "-t", 0], "ERROR: Number of trials must be greater than zero"),
        (["-m", "paired", "-a", a, "-o", out, "-j", meta, "--roi-permutations", 0],
         "ERROR: [-b, --directory-two] required in 'paired' group mode"),
    ]
    for args, message in cases:
        r = run_cli(monkeypatch, *args)
        assert r.output.strip().splitlines()[-1] == message, (args, r.output)
        assert not list(out.glob("region*"))


# ---- both files against numpy -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("saliency", [1, 2])
def test_two_directories_against_numpy(tmp_path, monkeypatch, golden, saliency):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "21")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    out = tmp_path / "out"
    ok(run_cli(monkeypatch, "-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta, "-s", saliency, "-w", W,
               "--roi-permutations", 12))
    g = golden("paired_synth_c30_c25_k18")
    x = np.concatenate([g["xa"], g["xb"]], axis=1)
    parts = np.array_split(np.arange(len(x)), 2)
    text, maxima = expected({"chr1": x[parts[0]], "chr2": x[parts[1]]}, (30, 25), saliency, 12, 21, "paired")
    check_outputs(out, "a_b_s%d" % saliency, text, maxima, 12)


@pytest.mark.parametrize("saliency", [1, 2])
@pytest.mark.parametrize("pair", [("a", "b"), ("a", "c")])          # a and c share biosamples 5-8
def test_compare_against_numpy(tmp_path, monkeypatch, saliency, pair):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "4")
    inp, gfile, meta, data = make_inputs(tmp_path)
    out = tmp_path / "out"
    ok(run_cli(monkeypatch, "-m", "paired", "-i", inp, "-o", out, "-j", meta, "--groups", gfile, "--compare",
               "%s:%s" % pair, "-s", saliency, "-w", W, "--roi-permutations", 7))
    cols = np.concatenate([np.asarray(COLUMNS[pair[0]]), np.asarray(COLUMNS[pair[1]])])
    files = {chrom: x[:, cols] for chrom, x in data.values()}
    sizes = (len(COLUMNS[pair[0]]), len(COLUMNS[pair[1]]))
    text, maxima = expected(files, sizes, saliency, 7, 4, "paired")
    check_outputs(out / ("%s_vs_%s" % pair), "%s_%s_s%d" % (pair + (saliency,)), text, maxima, 7)


@pytest.mark.parametrize("saliency", [1, 2])
@pytest.mark.parametrize("groups", [("g2", "g5", "g1"), ("g1", "g2", "g3", "g4", "g5")])
def test_multigroup_against_numpy(tmp_path, monkeypatch, saliency, groups):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "8")
    inp, _, meta, data = make_inputs(tmp_path)
    gfile = tmp_path / "mgroups.tsv"
    gfile.write_text(MGROUPS)
    out = tmp_path / "out"
    ok(run_cli(monkeypatch, "-m", "paired", "-i", inp, "-o", out, "-j", meta, "--groups", gfile, "--multigroup",
               ",".join(groups), "-s", saliency, "-w", W, "--roi-permutations", 6))
    cols = np.concatenate([np.asarray(MCOLS[g]) for g in groups])
    files = {chrom: x[:, cols] for chrom, x in data.values()}
    text, maxima = expected(files, [len(MCOLS[g]) for g in groups], saliency, 6, 8, "multigroup")
    name = "_".join(groups)
    check_outputs(out / name, "%s_s%d" % (name, saliency), text, maxima, 6)


# ---- every other output is unchanged ------------------------------------------------------------------------------------

@pytest.mark.parametrize("extra", [[], ["-n", "-t", "3", "-z", "150"], ["--null-permutations", "3"]])
def test_other_outputs_are_byte_identical(tmp_path, monkeypatch, golden, extra):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "5")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    common = ["-m", "paired", "-a", a, "-b", b, "-j", meta, "-s", 1, "-w", W, *extra]
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "plain"))
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "region", "--roi-permutations", 4))
    strip_region_files(tmp_path / "region", "a_b_s1")
    assert_same_outputs(tmp_path / "region", tmp_path / "plain")


def test_temp_files_equal_the_hand_over(tmp_path, monkeypatch):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "13")
    inp, _, meta, _ = make_inputs(tmp_path)
    gfile = tmp_path / "mgroups.tsv"
    gfile.write_text(MGROUPS + "x\t1-4\ny\t9-16\n")
    common = ["-m", "paired", "-i", inp, "-j", meta, "--groups", gfile, "-s", 2, "-w", W, "--multigroup", "g1,g3,g5",
              "--compare", "x:y", "--roi-permutations", 5]
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "mem"))
    monkeypatch.setenv("EPILOGOS_B200_KEEP_TEMP", "1")
    ok(run_cli(monkeypatch, *common, "-o", tmp_path / "files"))
    for d in ("g1_g3_g5", "x_vs_y"):
        assert_same_outputs(tmp_path / "files" / d, tmp_path / "mem" / d)


def test_roi_module_picks_the_temp_files_up(tmp_path, monkeypatch, golden):
    """The python -m stage entry points read temp_regionNull files and remove them."""
    from epilogos_b200 import expected as expected_stage, expectedCombination, roi_pairwise, scores, session
    monkeypatch.setenv("EPILOGOS_B200_SEED", "3")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    out = tmp_path / "out"; out.mkdir()
    be = RegionBackend()
    session.clear()
    pairs = [(f, b / f.name) for f in sorted(a.glob("*"))]
    for fa, fb in pairs:
        expected_stage.main(fa, fb, 18, 1, out, "t", 1, False, backend=be)
    expectedCombination.main(out, out / "exp_freq_t.npy", "t", False, backend=be)
    seed = region_seed(3)
    for fa, fb in pairs:
        scores.main(fa, fb, 18, 1, out, out / "exp_freq_t.npy", "t", 1, 17, -1, False, backend=be,
                    region_permutations=4, region_seed=seed, roi_width=W)
    assert len(list(out.glob("temp_regionNull_t_*.npz"))) == 2
    monkeypatch.setattr(session, "_backend", be)
    roi_pairwise.main(out, meta, "t", out / "exp_freq_t.npy", W, False)
    assert len((out / "regionPermutation_t.txt").read_text().splitlines()) > 0
    assert not list(out.glob("temp_*"))
    session.clear()


def test_score_stage_without_a_region_seed_raises(tmp_path, golden):
    from epilogos_b200 import pairwise
    a, b, _ = make_paired_inputs(tmp_path, golden)
    with pytest.raises(ValueError, match="region seed"):
        pairwise.calculateScoresPairwise(1, a / "x", b / "x", 18, tmp_path, tmp_path / "e.npy", "t", "x", 17, -1, False,
                                         backend=RegionBackend(), region_permutations=3)


def test_one_seed_per_run_without_a_fixed_seed(tmp_path, monkeypatch, golden):
    """Without EPILOGOS_B200_SEED every file must still use the same splits: the seed is drawn once per run."""
    monkeypatch.delenv("EPILOGOS_B200_SEED", raising=False)
    seeds = []

    class Spy(RegionBackend):
        def region_maxima_paired(self, *a, **k):
            seeds.append(a[6])
            return super().region_maxima_paired(*a, **k)
    a, b, meta = make_paired_inputs(tmp_path, golden, chroms=("chr1", "chr2", "chr3"))
    ok(run_cli(monkeypatch, "-m", "paired", "-a", a, "-b", b, "-o", tmp_path / "o", "-j", meta, "-w", W,
               "--roi-permutations", 2, backend=Spy()))
    assert len(seeds) == 3 and len(set(seeds)) == 1


def test_a_file_with_two_chromosomes_is_an_error(tmp_path, monkeypatch):
    inp, gfile, meta, data = make_inputs(tmp_path, files=(("chr1", 60),))
    x = data["epilogos_matrix_chr1.txt.gz"][1]
    path = inp / "epilogos_matrix_chr1.txt.gz"
    import gzip
    with gzip.open(path, "wt") as f:
        for r in range(len(x)):
            f.write("%s\t%d\t%d\t%s\n" % ("chr1" if r < 30 else "chr9", r * 200, r * 200 + 200,
                                          "\t".join(str(int(v) + 1) for v in x[r])))
    r = run_cli(monkeypatch, "-m", "paired", "-i", inp, "-o", tmp_path / "o", "-j", meta, "--groups", gfile,
                "--compare", "a:b", "-w", W, "--roi-permutations", 2)
    assert isinstance(r.exception, ValueError) and "epilogos_matrix_chr1.txt.gz" in str(r.exception)
    assert "one chromosome per input file" in str(r.exception)


def test_p_values_fall_as_window_sums_rise(tmp_path, monkeypatch, golden):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "6")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    out = tmp_path / "out"
    ok(run_cli(monkeypatch, "-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta, "-w", W, "--roi-permutations", 40))
    rows = [r.split("\t") for r in (out / "regionPermutation_a_b_s1.txt").read_text().splitlines()]
    s = [float(r[3]) for r in rows]
    k = [int(r[4]) for r in rows]
    assert len(set(k)) > 1
    for i in range(len(rows)):
        for j in range(len(rows)):
            if s[i] > s[j]:                 # the printed means are rounded: compare strictly larger ones
                assert k[i] <= k[j]
        assert rows[i][5] == "%.5e" % ((1.0 + k[i]) / 41.0)


# ---- the product's split draws and quantiser against the oracle ---------------------------------------------------------

@pytest.mark.parametrize("sizes,block", [((30, 25), 4), ((5, 5, 4), 3), ((64,), 1), ((40, 1, 90, 2), 7)])
def test_split_bitsets_are_the_oracle_permutations(sizes, block):
    from epilogos_b200 import region_null
    sizes = sizes if len(sizes) > 1 else (sizes[0], 1)
    P = 10
    N = sum(sizes)
    perms = list(ro.splits(77, N, P))
    got = []
    for p0, members in region_null.split_blocks(77, sizes, P, block):
        assert members.dtype == np.uint64 and members.shape[1:] == (len(sizes) - 1, (N + 63) // 64)
        got += [(p0 + i, m) for i, m in enumerate(members)]
    assert [p for p, _ in got] == list(range(P))
    edges = np.cumsum([0] + list(sizes))
    for p, m in got:
        bits = np.unpackbits(m.view(np.uint8), axis=1, bitorder="little")[:, :N]
        for g in range(len(sizes) - 1):
            assert sorted(np.flatnonzero(bits[g])) == sorted(perms[p][edges[g]:edges[g + 1]])


def test_quantiser_accepts_its_range_and_rejects_the_rest():
    from epilogos_b200 import region_null
    top = np.nextafter(2.0 ** 24, 0)
    assert region_null.quantise(np.array([0.0, -0.0, 2.0 ** -25, 3 * 2.0 ** -25, top])).tolist() == \
        [0, 0, 0, 2, int(np.rint(top * 2 ** 24))]
    for bad in (2.0 ** 24, np.nan, np.inf, -np.inf, -1e-30):
        with pytest.raises(ValueError, match="index 1"):
            region_null.quantise(np.array([1.0, bad]))


# ---- several ranks -----------------------------------------------------------------------------------------------------

GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
os.environ["EPILOGOS_B200_SHARD"] = {shard!r}
os.environ["EPILOGOS_B200_SEED"] = "17"
import torch.distributed as td
from test_region_permutations import RegionBackend
from epilogos_b200 import session, run
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size={world})
session._backend = RegionBackend()
run.main.main({args!r}, standalone_mode=False)
td.destroy_process_group()
"""


@pytest.mark.parametrize("shard,world", [("rows", 2), ("rows", 3), ("files", 2), ("files", 3)])
def test_gloo_ranks_equal_one(tmp_path, monkeypatch, shard, world):
    """Windows of 30 rows: in rows mode every rank holds fewer than W - 1 = 29 rows of chr3 (40 rows), so its windows
    run over the rows of the ranks after it."""
    monkeypatch.setenv("EPILOGOS_B200_SEED", "17")
    inp, _, meta, _ = make_inputs(tmp_path, files=(("chr1", 130), ("chr2", 70), ("chr3", 40)))
    gfile = tmp_path / "mgroups.tsv"
    gfile.write_text(MGROUPS)
    args = ["-m", "paired", "-i", str(inp), "-j", str(meta), "-s", "1", "-w", "30", "--groups", str(gfile),
            "--multigroup", "g1,g2,g4", "--compare", "g1:g5", "--roi-permutations", "5"]
    one = tmp_path / "one"
    ok(run_cli(monkeypatch, "-o", one, *args))
    many = tmp_path / "many"
    port = 38500 + (os.getpid() % 1500) + 11 * world + (5 if shard == "files" else 0)
    code = GLOO_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), shard=shard, port=port, world=world,
                              args=["-o", str(many)] + args)
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(world)]
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    for d in ("g1_g2_g4", "g1_vs_g5"):
        assert_same_outputs(many / d, one / d)
        assert (many / d / ("regionPermutation_%s_s1.txt" % d.replace("_vs_", "_"))).exists()
