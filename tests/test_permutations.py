"""Per-bin permutation p-values of paired mode (--null-permutations P) on a stand-in backend: the flag rules, the
pairwisePermutation file against a direct numpy computation, byte-identity of every other output, the temp-file route,
two gloo ranks, and --groups --compare.  The kernels are covered by test_permutations_gpu.py."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from click.testing import CliRunner

from oracle import epilogos_oracle as orc
from oracle import pairwise_stats_oracle as pso
from test_cli import META
from test_groups import GroupBackend, assert_same_outputs, make_inputs, subset_dir
from test_host_stages import ROOT
from test_pairwise_stats import make_paired_inputs, read_gz

TAG = "a_b_s1"


class PermBackend(GroupBackend):
    """The stand-in plus permutation_exceedances, built from its own shuffled_counts_device and scores."""

    def permutation_exceedances(self, cnt_a, cnt_b, dist, nperm, seed, size_a, size_b, width, bin_offset, saliency, exp,
                                score_widths, perms, exact=False, workspace_bytes=None):
        rows, k = cnt_a.shape
        oa, ob = self.shuffled_counts_device(cnt_a, cnt_b, size_a, size_b, seed, nperm, width=width, bin_offset=bin_offset)
        oa, ob = oa.reshape(-1, k), ob.reshape(-1, k)
        sa = self.scores(oa, score_widths[0], saliency, exp, perms=perms[0], exact=exact)
        sb = self.scores(ob, score_widths[1], saliency, exp, perms=perms[1], exact=exact)
        _, null = self.pairwise_combine(None, None, sa, sb)
        null = null.numpy().astype(np.float32).reshape(nperm, rows)
        counts = (np.abs(null) >= np.abs(np.asarray(dist, dtype=np.float32))).sum(axis=0).astype(np.uint32)
        return torch.from_numpy(counts.view(np.int32))


def run_cli(monkeypatch, *args, backend=None):
    from epilogos_b200 import run, session
    session.clear()
    monkeypatch.setattr(session, "_backend", backend or PermBackend())
    r = CliRunner().invoke(run.main, [str(a) for a in args])
    session.clear()
    return r


def paired(monkeypatch, a, b, meta, out, *extra):
    r = run_cli(monkeypatch, "-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta, "-s", 1, "-w", 9, *extra)
    assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)
    return r.output


def test_flag_rules_and_their_precedence(tmp_path, monkeypatch, golden):
    a, b, meta = make_paired_inputs(tmp_path, golden)
    out = tmp_path / "out"
    cases = [
        (["-i", a, "-o", out, "-j", meta, "--null-permutations", 5],
         "ERROR: [--null-permutations] requires [-m, --mode] 'paired'"),
        (["-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta, "--null-permutations", 0],
         "ERROR: Number of null permutations must be between 1 and 1000000"),
        (["-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta, "--null-permutations", 1000001],
         "ERROR: Number of null permutations must be between 1 and 1000000"),
        (["-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta, "--null-permutations", -3],
         "ERROR: Number of null permutations must be between 1 and 1000000"),
        # the existing rules keep their precedence
        (["-i", a, "-j", meta, "--null-permutations", 5], "ERROR: [-o, --output-directory] required"),
        (["-m", "paired", "-a", a, "-o", out, "-j", meta, "--null-permutations", 0],
         "ERROR: [-b, --directory-two] required in 'paired' group mode"),
        (["-m", "paired", "-a", a, "-b", b, "-o", out, "-j", meta, "-t", 0, "--null-permutations", 0],
         "ERROR: Number of trials must be greater than zero"),
    ]
    for args, message in cases:
        r = run_cli(monkeypatch, *args)
        assert r.output.strip().splitlines()[-1] == message, (args, r.output)
        assert not list(out.glob("pairwise*"))


def test_permutation_file_against_numpy(tmp_path, golden, monkeypatch):
    """Steps 1-4 on one file with the temp files kept between steps 3 and 4: the counts against numpy draws and scores,
    the file's columns against (1 + k) / (P + 1) and its Benjamini-Hochberg adjustment."""
    from epilogos_b200 import expected, expectedCombination, roi_pairwise, scores, session
    from epilogos_b200.pairwise import file_seed
    a, b, meta = make_paired_inputs(tmp_path, golden, chroms=("chr1",))
    out = tmp_path / "out"; out.mkdir()
    be = PermBackend()
    session.clear()
    fa, fb = a / "epilogos_matrix_chr1.txt.gz", b / "epilogos_matrix_chr1.txt.gz"
    expected.main(fa, fb, 18, 1, out, "t", 1, False, backend=be)
    expectedCombination.main(out, out / "exp_freq_t.npy", "t", False, backend=be)
    exp = np.load(out / "exp_freq_t.npy")
    monkeypatch.setenv("EPILOGOS_B200_SEED", "11")
    P = 9
    scores.main(fa, fb, 18, 1, out, out / "exp_freq_t.npy", "t", 1, 17, -1, False, backend=be, permutations=P)
    z = np.load(out / "temp_permutations_t_epilogos_matrix_chr1.npz")
    assert z["exceedances"].dtype == np.uint32 and int(z["permutations"]) == P and str(z["chrName"][0]) == "chr1"
    null = np.load(out / "temp_nullDistances_t_epilogos_matrix_chr1.npz")["nullDistances"]

    xa, xb = golden("paired_synth_c30_c25_k18")["xa"], golden("paired_synth_c30_c25_k18")["xb"]
    ca, cb = orc.bin_counts(xa, 18).astype(np.int64), orc.bin_counts(xb, 18).astype(np.int64)
    seed = file_seed(11, "epilogos_matrix_chr1")
    nulls = []
    for p in range(P):
        ga = np.zeros_like(ca); gb = np.zeros_like(cb)
        for r in range(len(ca)):
            rng = np.random.default_rng([seed & (2 ** 63 - 1), p, r])
            comb = ca[r] + cb[r]
            ga[r] = rng.multivariate_hypergeometric(comb, min(30, int(comb.sum())))
            rest = comb - ga[r]
            gb[r] = rng.multivariate_hypergeometric(rest, min(25, int(rest.sum())))
        d = orc.s1_scores_from_counts(ga, 30, exp) - orc.s1_scores_from_counts(gb, 25, exp)
        nulls.append(np.sum(np.square(d), axis=1) * np.sign(np.sum(d, axis=1)))
    nulls = np.array(nulls, dtype=np.float32)
    assert nulls[0].tobytes() == null.tobytes()            # permutation 0 is the run's own null
    txt = read_gz(out / "pairwiseDelta_t_epilogos_matrix_chr1.txt.gz").splitlines()
    delta = np.array([[float(v) for v in l.split("\t")[3:]] for l in txt]).astype(np.float32)
    dist, _ = orc.paired_real_reductions(delta, round_trip=False)
    k = (np.abs(nulls) >= np.abs(np.asarray(dist, dtype=np.float32))).sum(axis=0)
    assert z["exceedances"].tolist() == k.tolist()
    assert k.max() > 0 and k.min() < P

    roi_pairwise.main(out, meta, "t", out / "exp_freq_t.npy", 9, False, backend=be)
    pv = (k + 1.0) / (P + 1.0)
    q = pso.bh(pv)
    want = "".join("%s\t%s\t%s\t%d\t%.5e\t%.5e\n" % (*l.split("\t")[:3], k[i], pv[i], q[i]) for i, l in enumerate(txt))
    assert read_gz(out / "pairwisePermutation_t.txt.gz") == want
    assert not list(out.glob("temp_*"))
    session.clear()


@pytest.mark.parametrize("extra", [[], ["-n", "-t", "3", "-z", "150"], ["-g", "20", "-q", "0"]])
def test_other_outputs_are_byte_identical_with_and_without_the_flag(tmp_path, golden, monkeypatch, extra):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "5")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    plain, perm = tmp_path / "plain", tmp_path / "perm"
    paired(monkeypatch, a, b, meta, plain, *extra)
    paired(monkeypatch, a, b, meta, perm, *extra, "--null-permutations", 4)
    name = "pairwisePermutation_%s.txt.gz" % TAG
    rows = read_gz(perm / name).splitlines()
    assert len(rows) == len(read_gz(perm / ("pairwiseMetrics_%s.txt.gz" % TAG)).splitlines())
    assert {int(r.split("\t")[3]) for r in rows} <= set(range(5))
    (perm / name).unlink()
    assert_same_outputs(perm, plain)


@pytest.mark.parametrize("null_mode", ["device", "reference"])
def test_temp_file_route_equals_the_hand_over(tmp_path, golden, monkeypatch, null_mode):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "8")
    monkeypatch.setenv("EPILOGOS_B200_NULL", null_mode)
    a, b, meta = make_paired_inputs(tmp_path, golden)
    mem, disk = tmp_path / "mem", tmp_path / "disk"
    np.random.seed(2)
    paired(monkeypatch, a, b, meta, mem, "-n", "-t", "3", "-z", "150", "--null-permutations", 6)
    monkeypatch.setenv("EPILOGOS_B200_KEEP_TEMP", "1")
    np.random.seed(2)
    paired(monkeypatch, a, b, meta, disk, "-n", "-t", "3", "-z", "150", "--null-permutations", 6)
    assert_same_outputs(disk, mem)
    assert not list(disk.glob("temp_*"))


def test_roi_pairwise_module_picks_the_temp_files_up(tmp_path, golden, monkeypatch):
    """roi_pairwise.main (what python -m epilogos_b200.roi_pairwise runs) on a directory of step 1-3 outputs of several
    files writes the permutation file with no new argument, and removes the temp files."""
    from epilogos_b200 import expected, expectedCombination, roi_pairwise, scores, session
    a, b, meta = make_paired_inputs(tmp_path, golden)
    out = tmp_path / "out"; out.mkdir()
    be = PermBackend()
    session.clear()
    monkeypatch.setenv("EPILOGOS_B200_SEED", "3")
    pairs = [(f, b / f.name) for f in sorted(a.glob("*"))]
    for fa, fb in pairs:
        expected.main(fa, fb, 18, 1, out, "t", 1, False, backend=be)
    expectedCombination.main(out, out / "exp_freq_t.npy", "t", False, backend=be)
    for fa, fb in pairs:
        scores.main(fa, fb, 18, 1, out, out / "exp_freq_t.npy", "t", 1, 17, -1, False, backend=be, permutations=3)
    assert len(list(out.glob("temp_permutations_t_*.npz"))) == 2
    monkeypatch.setattr(session, "_backend", be)
    roi_pairwise.main(out, meta, "t", out / "exp_freq_t.npy", 9, False)
    rows = read_gz(out / "pairwisePermutation_t.txt.gz").splitlines()
    assert [r.split("\t")[0] for r in rows] == [r.split("\t")[0] for r in read_gz(out / "pairwiseMetrics_t.txt.gz").splitlines()]
    assert not list(out.glob("temp_*"))
    session.clear()


GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
os.environ["EPILOGOS_B200_SHARD"] = {shard!r}
os.environ["EPILOGOS_B200_SEED"] = "31"
import torch.distributed as td
from pathlib import Path
from test_permutations import PermBackend
from epilogos_b200 import dist, run
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
out = Path({out!r}); a = Path({a!r}); b = Path({b!r})
pairs = [(f, b / f.name) for f in sorted(a.glob("*"))]
say = (lambda *x, **k: print(*x, **k, flush=True)) if dist.rank() == 0 else (lambda *x, **k: None)
run.run_stages(pairs, "paired", 18, 1, out, "a_b_s1", out / "exp_freq_a_b_s1.npy", 1, 17, -1, {meta!r}, 9, False, say,
               backend=PermBackend(), permutations=5)
td.destroy_process_group()
"""


@pytest.mark.parametrize("shard", ["rows", "files"])
def test_two_gloo_ranks_write_the_same_permutation_file_as_one(tmp_path, golden, monkeypatch, shard):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "31")
    a, b, meta = make_paired_inputs(tmp_path, golden)
    one = tmp_path / "one"
    paired(monkeypatch, a, b, meta, one, "--null-permutations", 5)
    two = tmp_path / "two"; two.mkdir()
    port = 36600 + (os.getpid() % 2000) + (7 if shard == "files" else 0)
    code = GLOO_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), shard=shard, port=port, out=str(two), a=str(a),
                              b=str(b), meta=str(meta))
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    for name in ("pairwisePermutation_%s.txt.gz" % TAG, "pairwiseMetrics_%s.txt.gz" % TAG):
        assert read_gz(one / name) == read_gz(two / name), name
    assert not list(two.glob("temp_*"))


def test_groups_compare_equals_the_two_directory_run(tmp_path, monkeypatch):
    monkeypatch.setenv("EPILOGOS_B200_SEED", "23")
    inp, gfile, meta, data = make_inputs(tmp_path)
    out = tmp_path / "out"
    common = ["-j", meta, "-s", 2, "-w", 9, "--null-permutations", 7]
    r = run_cli(monkeypatch, "-m", "paired", "-i", inp, "-o", out, "--groups", gfile, "--compare", "a:b",
                "--compare", "c:u", *common)
    assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)
    for ga, gb in (("a", "b"), ("c", "u")):
        got = out / ("%s_vs_%s" % (ga, gb))
        want = tmp_path / "want" / got.name
        r = run_cli(monkeypatch, "-m", "paired", "-a", subset_dir(tmp_path, data, ga), "-b", subset_dir(tmp_path, data, gb),
                    "-o", want, *common)
        assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)
        assert_same_outputs(got, want)
        assert (got / ("pairwisePermutation_%s_%s_s2.txt.gz" % (ga, gb))).exists()
