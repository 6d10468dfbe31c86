"""Host-side stage drivers (epilogos_b200.expected / expectedCombination / scores) on CPU.

The compute provider is replaced by tests/fake_backend.OracleBackend so that what is tested here is the host
logic: row sharding, all-reduce of the integer tables, gather of score rows, file names / dtypes / text format
-- at world size 1 and at world size 2 over gloo.  The CUDA provider is exercised by the -m gpu tests.
"""
import gzip
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def write_tsv(path, x0, chrom="chr1", gz=False):
    opener = gzip.open if gz else open
    with opener(path, "wt") as f:
        for r in range(x0.shape[0]):
            f.write("%s\t%d\t%d\t%s\n" % (chrom, r * 200, r * 200 + 200, "\t".join(str(int(v) + 1) for v in x0[r])))


def run_single_pipeline(tmp, x, k, saliency, backend, gz=False):
    from epilogos_b200 import expected, expectedCombination, scores, session
    session.clear()
    inp = tmp / "in"; out = tmp / "out"
    inp.mkdir(exist_ok=True); out.mkdir(exist_ok=True)
    f = inp / ("epilogos_matrix_chr1.txt" + (".gz" if gz else ""))
    write_tsv(f, x, gz=gz)
    tag = "in_s%d" % saliency
    expected.main(f, "null", k, saliency, out, tag, 1, False, backend=backend)
    temp = out / ("temp_exp_freq_%s_epilogos_matrix_chr1.npy" % tag)
    counts = np.load(temp)
    exp_path = out / ("exp_freq_%s.npy" % tag)
    expectedCombination.main(out, exp_path, tag, False, backend=backend)
    assert not temp.exists()
    scores.main(f, "null", k, saliency, out, exp_path, tag, 1, k - 1, -1, False, backend=backend)
    npz = np.load(out / ("temp_scores_%s_epilogos_matrix_chr1.npz" % tag), allow_pickle=True)
    with gzip.open(out / ("scores_%s_epilogos_matrix_chr1.txt.gz" % tag), "rb") as g:
        text = g.read()
    return counts, np.load(exp_path), npz, text


def test_helpers_rows_and_parse(tmp_path, golden):
    from epilogos_b200 import helpers
    x = golden("real10_chr1_k18")["x"][:257]
    f = tmp_path / "m.txt.gz"
    write_tsv(f, x, gz=True)
    assert helpers.countRows(f) == 257
    assert helpers.splitRows(257, 3) == [(0, 85), (85, 171), (171, 257)]
    loc, s0 = helpers.read_matrix(f)
    assert s0.dtype == np.int8 and np.array_equal(s0, x)
    assert loc["chrom"][0] == "chr1" and loc["start"][5] == 1000 and loc["end"][-1] == 257 * 200
    _, part = helpers.read_matrix(f, rows=(85, 171), want_locations=False)
    assert np.array_equal(part, x[85:171])
    assert helpers.strToBool("True") is True and helpers.strToBool("False") is False
    with pytest.raises(ValueError):
        helpers.strToBool("yes")


@pytest.mark.parametrize("saliency", [1, 2])
def test_single_pipeline_files_match_reference(tmp_path, golden, saliency):
    from fake_backend import OracleBackend
    g = golden("real10_chr1_k18")
    x = g["x"]
    counts, exp, npz, text = run_single_pipeline(tmp_path, x, 18, saliency, OracleBackend(), gz=(saliency == 2))
    assert counts.dtype == np.int64 and np.array_equal(counts, g["s%d_counts" % saliency])
    assert exp.dtype == np.float32 and exp.tobytes() == g["s%d_exp" % saliency].tobytes()
    assert npz["scoreArr"].dtype == np.float32
    assert npz["scoreArr"].tobytes() == g["s%d_scores" % saliency].tobytes()
    assert str(npz["chrName"][0]) == "chr1" and npz["locationArr"].shape == (x.shape[0], 3)
    assert text == g["s%d_text" % saliency].tobytes()


def test_prefetch_parses_every_file_once_and_stages_reuse_it(tmp_path, golden, monkeypatch):
    """session.prefetch (what the CLI calls before STEP 1): all files of a directory are parsed concurrently, once; the
    expected and the score stage of every file find their shard in the cache (no second parse), and the multi-file
    table equals the table of the concatenated matrix (expectedCombination.py:30-35)."""
    from fake_backend import OracleBackend
    from epilogos_b200 import expected, expectedCombination, helpers, scores, session
    from oracle import epilogos_oracle as orc
    session.clear()
    x = golden("real10_chr1_k18")["x"]
    parts = [x[:700], x[700:1500], x[1500:2100], x[2100:2600], x[2600:3000], x[3000:3300]]
    inp = tmp_path / "in"; out = tmp_path / "out"
    inp.mkdir(); out.mkdir()
    files = []
    for i, part in enumerate(parts):
        f = inp / ("epilogos_matrix_chr%d.txt.gz" % (i + 1))
        write_tsv(f, part, chrom="chr%d" % (i + 1), gz=True)
        files.append(f)
    be = OracleBackend()
    calls = []
    real = helpers.read_matrix
    monkeypatch.setattr(helpers, "read_matrix", lambda *a, **k: (calls.append(str(a[0])), real(*a, **k))[1])
    session.prefetch([(f, "null") for f in files], 18, backend=be, workers=3)
    assert sorted(calls) == sorted(str(f) for f in files)
    for f in files:
        expected.main(f, "null", 18, 2, out, "t", 1, False, backend=be)
    exp_path = out / "exp_freq_t.npy"
    expectedCombination.main(out, exp_path, "t", False, backend=be)
    for f in files:
        scores.main(f, "null", 18, 2, out, exp_path, "t", 1, 17, -1, False, backend=be)
    assert len(calls) == len(files)                                   # nothing was parsed twice
    whole = np.concatenate(parts)
    assert np.load(exp_path).tobytes() == orc.normalize_expected(orc.s2_expected_counts(whole, 18)).tobytes()
    got = np.concatenate([np.load(out / ("temp_scores_t_epilogos_matrix_chr%d.npz" % (i + 1)), allow_pickle=True)["scoreArr"]
                          for i in range(len(parts))])
    assert got.tobytes() == orc.s2_scores(whole, 18, np.load(exp_path)).tobytes()
    session.clear()


def test_simsearch_region_start_lookup():
    """similaritySearch_calc.py:107-109: the first genome row whose chromosome AND start match, // blockSize -- with
    chromosomes whose coordinates restart, a chromosome that appears in two separate runs, and unsorted starts."""
    from epilogos_b200.similaritySearch_calc import _region_starts
    chrom = np.array(["chr1"] * 6 + ["chr2"] * 5 + ["chr1"] * 3 + ["chrX"] * 4, dtype=object)
    start = np.array([0, 200, 400, 600, 800, 1000, 0, 200, 400, 600, 800, 5000, 5200, 5400, 600, 200, 400, 0])
    coords = np.empty((len(chrom), 3), dtype=object)
    coords[:, 0], coords[:, 1], coords[:, 2] = chrom, start, start + 200
    rois = np.array([["chr1", 400, 0], ["chr2", 400, 0], ["chr1", 5200, 0], ["chrX", 200, 0], ["chr2", 0, 0]], dtype=object)
    want = [int(np.flatnonzero((chrom == c) & (start == s))[0]) for c, s, _ in rois]
    assert _region_starts(coords, rois, 1).tolist() == want == [2, 8, 12, 15, 6]
    assert _region_starts(coords, rois, 5).tolist() == [w // 5 for w in want]
    with pytest.raises(IndexError):
        _region_starts(coords, np.array([["chr2", 5000, 0]], dtype=object), 1)


def test_bad_saliency_raises(tmp_path):
    from fake_backend import OracleBackend
    from epilogos_b200 import expected
    f = tmp_path / "m.txt"
    write_tsv(f, np.zeros((4, 3), dtype=np.int8))
    with pytest.raises(ValueError):
        expected.main(f, "null", 18, 4, tmp_path, "t", 1, False, backend=OracleBackend())


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import numpy as np, torch.distributed as dist
from pathlib import Path
from fake_backend import OracleBackend
from epilogos_b200 import expected, expectedCombination, scores
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
out = Path({out!r}); f = Path({f!r}); be = OracleBackend()
for s in (1, 2):
    tag = "in_s%d" % s
    expected.main(f, "null", 18, s, out, tag, 1, False, backend=be)
    expectedCombination.main(out, out / ("exp_freq_%s.npy" % tag), tag, False, backend=be)
    scores.main(f, "null", 18, s, out, out / ("exp_freq_%s.npy" % tag), tag, 1, 17, -1, False, backend=be)
dist.destroy_process_group()
"""


def test_world_size_two_gloo_matches_single_rank(tmp_path, golden):
    g = golden("real10_chr1_k18")
    x = g["x"][:1001]                       # odd row count: uneven shards
    f = tmp_path / "epilogos_matrix_chr1.txt"
    write_tsv(f, x)
    out = tmp_path / "out"
    out.mkdir()
    port = 29500 + (os.getpid() % 2000)
    code = WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), port=port, out=str(out), f=str(f))
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=300)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    from oracle import epilogos_oracle as orc
    for s in (1, 2):
        tag = "in_s%d" % s
        counts = orc.s1_expected_counts(x, 18) if s == 1 else orc.s2_expected_counts(x, 18)
        exp = np.load(out / ("exp_freq_%s.npy" % tag))
        assert exp.tobytes() == orc.normalize_expected(counts).tobytes()
        ref = orc.s1_scores(x, 18, exp) if s == 1 else orc.s2_scores(x, 18, exp)
        npz = np.load(out / ("temp_scores_%s_epilogos_matrix_chr1.npz" % tag), allow_pickle=True)
        assert npz["scoreArr"].tobytes() == ref.tobytes()
        with gzip.open(out / ("scores_%s_epilogos_matrix_chr1.txt.gz" % tag), "rb") as gzf:
            text = gzf.read()
        starts = np.arange(x.shape[0]) * 200
        assert text == orc.format_scores_text(ref, "chr1", starts, starts + 200)


def run_paired_pipeline(tmp, xa, xb, k, saliency, backend, seed, group_size=-1, quiescent=None, null_mode="reference"):
    from epilogos_b200 import expected, expectedCombination, scores, session
    session.clear()
    a = tmp / "a"; b = tmp / "b"; out = tmp / "out"
    for d in (a, b, out):
        d.mkdir(exist_ok=True)
    fa, fb = a / "epilogos_matrix_chr1.txt", b / "epilogos_matrix_chr1.txt"
    write_tsv(fa, xa); write_tsv(fb, xb)
    tag = "a_b_s%d" % saliency
    expected.main(fa, fb, k, saliency, out, tag, 1, False, backend=backend)
    counts = np.load(out / ("temp_exp_freq_%s_epilogos_matrix_chr1.npy" % tag))
    exp_path = out / ("exp_freq_%s.npy" % tag)
    expectedCombination.main(out, exp_path, tag, False, backend=backend)
    os.environ["EPILOGOS_B200_NULL"] = null_mode
    np.random.seed(seed)
    try:
        scores.main(fa, fb, k, saliency, out, exp_path, tag, 1, k - 1 if quiescent is None else quiescent, group_size,
                    False, backend=backend)
    finally:
        os.environ.pop("EPILOGOS_B200_NULL", None)
    null = np.load(out / ("temp_nullDistances_%s_epilogos_matrix_chr1.npz" % tag))["nullDistances"]
    quies = np.load(out / ("temp_quiescence_%s_epilogos_matrix_chr1.npz" % tag))["quiescenceArr"]
    with gzip.open(out / ("pairwiseDelta_%s_epilogos_matrix_chr1.txt.gz" % tag), "rb") as g:
        text = g.read()
    return counts, np.load(exp_path), null, quies, text


@pytest.mark.parametrize("name", ["paired_real10_k18", "paired_synth_g20_k18", "paired_synth_q0_k18",
                                  "paired_synth_g40_k18"])
def test_paired_pipeline_files_match_reference(tmp_path, golden, name):
    from fake_backend import OracleBackend
    g = golden(name)
    for s in (1, 2):
        if "s%d_counts" % s not in g.files:
            continue
        sub = tmp_path / ("s%d" % s)
        sub.mkdir()
        counts, exp, null, quies, text = run_paired_pipeline(sub, g["xa"], g["xb"], int(g["num_states"]), s,
                                                             OracleBackend(), int(g["seed"]), int(g["group_size"]),
                                                             int(g["quiescent_state"]))
        assert np.array_equal(counts, g["s%d_counts" % s]) and exp.tobytes() == g["s%d_exp" % s].tobytes()
        assert null.dtype == np.float32 and null.tobytes() == g["s%d_null" % s].tobytes()
        assert quies.dtype == np.bool_ and np.array_equal(quies, g["s%d_quiescence" % s])
        assert text == g["s%d_delta_text" % s].tobytes()


FILES_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
os.environ["EPILOGOS_B200_SHARD"] = {shard!r}.split("-")[0]
if {shard!r}.endswith("-redundant"):
    os.environ["EPILOGOS_B200_READ"] = "redundant"
import torch.distributed as td
from pathlib import Path
from fake_backend import OracleBackend
from epilogos_b200 import dist, helpers, run
_read, _parsed = helpers.read_matrix, []
def _counting(path, *a, **k):
    _parsed.append(Path(path).name)
    return _read(path, *a, **k)
helpers.read_matrix = _counting
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
out = Path({out!r}); inp = Path({inp!r})
pairs = [(f, "null") for f in sorted(inp.glob("*"))]
lead = dist.rank() == 0
say = (lambda *a, **k: print(*a, **k, flush=True)) if lead else (lambda *a, **k: None)
run.run_stages(pairs, "single", 18, 2, out, "in_s2", out / "exp_freq_in_s2.npy", 1, 17, -1, {meta!r}, 20, False, say,
               backend=OracleBackend())
print("RANK", td.get_rank(), "files", sorted(p.name for p in out.glob("scores_*")), flush=True)
print("PARSED", td.get_rank(), " ".join(_parsed), flush=True)
td.destroy_process_group()
"""


@pytest.mark.parametrize("shard", ["files", "rows", "rows-redundant"])
def test_run_stages_world_size_two_files_or_rows(tmp_path, golden, shard):
    """run.run_stages on two gloo ranks with three input files of different sizes: whole files dealt to the ranks
    (EPILOGOS_B200_SHARD=files: each rank runs the unsharded stages on its files, tables meet through the files) and rows
    split over the ranks (default: every file is parsed by ONE rank, which deals the row ranges to the others;
    EPILOGOS_B200_READ=redundant: every rank parses every file) all reproduce the single-rank result -- table, every score
    file, ROI list."""
    from oracle import epilogos_oracle as orc
    from test_cli import META
    g = golden("real10_chr1_k18")
    x = g["x"]
    parts = {"epilogos_matrix_chr1": x[:1700], "epilogos_matrix_chr2": x[1700:2300], "epilogos_matrix_chrX": x[2300:3301]}
    inp = tmp_path / "in"; out = tmp_path / "out"
    inp.mkdir(); out.mkdir()
    for name, part in parts.items():
        write_tsv(inp / (name + ".txt"), part, chrom=name.split("_")[-1])
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    port = 31500 + (os.getpid() % 2000) + (7 if shard == "files" else 0)
    code = FILES_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), port=port, out=str(out), inp=str(inp),
                               meta=str(meta), shard=shard)
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=300)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    if shard == "files":
        assert "Input files dealt to the ranks: 3 files over 2 GPUs" in logs[0]
    parsed = [line.split()[2:] for log in logs for line in log.splitlines() if line.startswith("PARSED")]
    assert len(parsed) == 2
    names = sorted(n for p in parsed for n in p)
    if shard == "rows-redundant":
        assert names == sorted(2 * [n + ".txt" for n in parts])                  # every rank parsed every file
    else:
        assert names == sorted(n + ".txt" for n in parts)                        # every file parsed exactly once, by one rank
        assert all(len(p) >= 1 for p in parsed)                                   # ... and both ranks read something
    allx = np.concatenate(list(parts.values()))
    exp = orc.normalize_expected(orc.s2_expected_counts(allx, 18))
    for name, part in parts.items():
        ref = orc.s2_scores(part, 18, exp)
        with gzip.open(out / ("scores_in_s2_%s.txt.gz" % name), "rb") as gzf:
            text = gzf.read()
        starts = np.arange(part.shape[0]) * 200
        assert text == orc.format_scores_text(ref, name.split("_")[-1], starts, starts + 200)
    # step 4 ran once, on rank 0, over every file's scores, and cleaned up
    assert (out / "regionsOfInterest_in_s2.txt").exists() and not list(out.glob("temp_*")) and not (out / "exp_freq_in_s2.npy").exists()
    assert len((out / "regionsOfInterest_in_s2.txt").read_text().splitlines()) > 10


BAD_INPUT_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import torch.distributed as td
from fake_backend import OracleBackend
from epilogos_b200 import session
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
try:
    session.load_shard({f!r}, "null", 18, OracleBackend())
    print("NO ERROR", flush=True)
except Exception as exc:
    print("RAISED", td.get_rank(), type(exc).__name__, str(exc), flush=True)
td.destroy_process_group()
"""


def test_unreadable_input_fails_on_every_rank_when_one_rank_reads(tmp_path):
    """Rows mode with one reader per file: a file the reader cannot parse (label outside 1..numStates) raises on BOTH
    ranks -- the reader tells the waiting rank instead of leaving it in the exchange."""
    f = tmp_path / "epilogos_matrix_chr1.txt"
    f.write_text("".join("chr1\t%d\t%d\t1\t2\t%d\n" % (i * 200, i * 200 + 200, 19 if i == 7 else 3) for i in range(20)))
    port = 33500 + (os.getpid() % 2000)
    code = BAD_INPUT_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), port=port, f=str(f))
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=120)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    raised = [line for log in logs for line in log.splitlines() if line.startswith("RAISED")]
    assert len(raised) == 2 and all("row 7" in line and "outside 1..18" in line for line in raised), logs


def test_deal_files_balances_by_size(tmp_path):
    from epilogos_b200 import run
    sizes = {"a": 900, "b": 500, "c": 400, "d": 300, "e": 100}
    pairs = []
    for n, s in sizes.items():
        (tmp_path / n).write_bytes(b"x" * s)
        pairs.append((tmp_path / n, "null"))
    dealt = run.deal_files(pairs, 2)
    loads = [sum(sizes[p[0].name] for p in part) for part in dealt]
    assert sorted(p[0].name for part in dealt for p in part) == sorted(sizes) and abs(loads[0] - loads[1]) <= 200
    assert run.deal_files(pairs, 2) == dealt                   # deterministic: every rank computes the same deal


def test_readStates_shim_matches_the_reference_conventions(tmp_path):
    """helpers.readStates (the reference's name and return convention): row ranges, 0-based int arrays, the paired
    concatenation, and the seeded shuffle equal to the oracle's restatement of helpers.py:183-194."""
    from epilogos_b200 import helpers
    from oracle import epilogos_oracle as orc
    xa = orc.synth_states(40, 7, 18, seed=1)
    xb = orc.synth_states(40, 5, 18, seed=2)
    fa, fb = tmp_path / "a.txt", tmp_path / "b.txt.gz"
    write_tsv(fa, xa)
    write_tsv(fb, xb, gz=True)
    got = helpers.readStates(fa, rowsToCalc=(3, 31), verbose=False)
    assert got.dtype == np.dtype(int) and np.array_equal(got, xa[3:31])
    both = helpers.readStates(fa, fb, (0, 40), expBool=True, verbose=False)
    assert np.array_equal(both, np.concatenate((xa, xb), axis=1))
    for group in (-1, 4):
        np.random.seed(123)
        a, b, sa, sb = helpers.readStates(fa, fb, (5, 25), expBool=False, verbose=False, groupSize=group)
        perm = orc.reference_shuffle_indices(123, 20, 12)
        wa, wb = orc.paired_split(xa[5:25], xb[5:25], perm, group)[-2:]
        assert np.array_equal(a, xa[5:25]) and np.array_equal(b, xb[5:25])
        assert np.array_equal(sa, wa) and np.array_equal(sb, wb)


def test_expected_chunk_workers_under_the_reference_names(tmp_path):
    """expected.s1Calc / s2Calc (the reference's per-chunk workers, expected.py:90-162) on a row range, single and paired."""
    from epilogos_b200 import expected
    from fake_backend import OracleBackend
    from oracle import epilogos_oracle as orc
    xa = orc.synth_states(60, 9, 18, seed=3)
    xb = orc.synth_states(60, 6, 18, seed=4)
    fa, fb = tmp_path / "a.txt", tmp_path / "b.txt"
    write_tsv(fa, xa)
    write_tsv(fb, xb)
    be = OracleBackend()
    n1 = expected.s1Calc(fa, "null", (10, 50), 18, False, backend=be)
    n2 = expected.s2Calc(fa, "null", (10, 50), 18, False, backend=be)
    assert n1.dtype == np.int64 and np.array_equal(n1, orc.s1_expected_counts_rowloop(xa[10:50], 18))
    assert n2.dtype == np.int64 and np.array_equal(n2, orc.s2_expected_counts_rowloop(xa[10:50], 18))
    both = np.concatenate((xa, xb), axis=1)
    assert np.array_equal(expected.s2Calc(fa, fb, (0, 60), 18, False, backend=be), orc.s2_expected_counts(both, 18))


NPERM_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import torch.distributed as td
from pathlib import Path
from fake_backend import OracleBackend
from epilogos_b200 import pairwise, session
td.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
pairwise.calculateScoresPairwise(1, Path({fa!r}), Path({fb!r}), 18, Path({out!r}), Path({exp!r}), "t", "m", 17, -1, False,
                                 backend=OracleBackend(), null_mode="device", seed=4242, nperm=3)
td.destroy_process_group()
"""


def test_device_null_nperm_rows_are_permutations_and_do_not_depend_on_sharding(tmp_path):
    """Device-drawn null with nperm > 1: nullDistances is [nperm, rows] with row p = the p-th shuffle of every bin (checked
    against a direct evaluation of the same keyed draws), and two ranks sharing the rows produce the same array as one
    rank, because a bin's draw is keyed by (seed, file, permutation, GLOBAL bin index)."""
    from fake_backend import OracleBackend
    from epilogos_b200 import pairwise, session
    from oracle import epilogos_oracle as orc
    xa = orc.synth_states(37, 9, 18, seed=21)
    xb = orc.synth_states(37, 6, 18, seed=22)
    fa, fb = tmp_path / "a.txt", tmp_path / "b.txt"
    write_tsv(fa, xa); write_tsv(fb, xb)
    exp = orc.normalize_expected(orc.s1_expected_counts(np.concatenate((xa, xb), axis=1), 18))
    exp_path = tmp_path / "exp.npy"
    np.save(exp_path, exp)
    be = OracleBackend()
    one = tmp_path / "one"; one.mkdir()
    session.clear()
    pairwise.calculateScoresPairwise(1, fa, fb, 18, one, exp_path, "t", "m", 17, -1, False, backend=be,
                                     null_mode="device", seed=4242, nperm=3)
    null1 = np.load(one / "temp_nullDistances_t_m.npz")["nullDistances"]
    assert null1.shape == (3, 37) and null1.dtype == np.float32
    # direct evaluation of permutation p from the same keyed draws
    ca, cb = be.counts(xa, 18), be.counts(xb, 18)
    oa, ob = be.shuffled_counts_device(ca, cb, 9, 6, pairwise.file_seed(4242, "m"), nperm=3, width=15)
    for p in range(3):
        na = orc.s1_scores_from_counts(be._cnt(oa[p]), 9, exp)
        nb = orc.s1_scores_from_counts(be._cnt(ob[p]), 6, exp)
        d = na - nb
        want = np.sum(np.square(d), axis=1) * np.sign(np.sum(d, axis=1))
        assert null1[p].tobytes() == want.astype(np.float32).tobytes()
    assert not np.array_equal(null1[0], null1[1])
    # another file name -> another stream
    other = tmp_path / "other"; other.mkdir()
    session.clear()
    pairwise.calculateScoresPairwise(1, fa, fb, 18, other, exp_path, "t", "m2", 17, -1, False, backend=be,
                                     null_mode="device", seed=4242, nperm=3)
    assert not np.array_equal(np.load(other / "temp_nullDistances_t_m2.npz")["nullDistances"], null1)
    # two gloo ranks sharing the rows
    two = tmp_path / "two"; two.mkdir()
    port = 33500 + (os.getpid() % 2000)
    code = NPERM_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), port=port, fa=str(fa), fb=str(fb), out=str(two),
                               exp=str(exp_path))
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    logs = [p.communicate(timeout=300)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    null2 = np.load(two / "temp_nullDistances_t_m.npz")["nullDistances"]
    assert null2.tobytes() == null1.tobytes()
    session.clear()


def test_shuffled_widths_follow_numpy_slicing():
    from epilogos_b200.pairwise import shuffled_widths
    for c1, c2, g in [(30, 25, -1), (30, 25, 20), (30, 25, 40), (30, 25, 55), (30, 25, 70), (5, 5, 5)]:
        sh = np.zeros((1, c1 + c2))
        want = (c1, c2) if g == -1 else (sh[:, :g].shape[1], sh[:, g:2 * g].shape[1])
        assert shuffled_widths(c1, c2, g) == want


@pytest.mark.parametrize("shard", ["rows", "files"])
def test_run_stages_world_size_eight(tmp_path, shard):
    """The 8-GPU shape of the CLI on gloo: eight ranks, eight input files of different sizes (some shorter than the world
    size times a few rows), rows split over the ranks or whole files dealt to them -- every score file equals the
    single-process oracle result for the table of ALL files, and step 4 runs once."""
    from oracle import epilogos_oracle as orc
    from test_cli import META
    parts = {"epilogos_matrix_chr%d" % (i + 1): orc.synth_states(90 + 37 * i, 40, 18, seed=i) for i in range(8)}
    inp = tmp_path / "in"; out = tmp_path / "out"
    inp.mkdir(); out.mkdir()
    for name, part in parts.items():
        write_tsv(inp / (name + ".txt"), part, chrom=name.split("_")[-1])
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    port = 35500 + (os.getpid() % 2000) + (11 if shard == "files" else 0)
    code = FILES_WORKER.format(root=str(ROOT), tests=str(ROOT / "tests"), port=port, out=str(out), inp=str(inp),
                               meta=str(meta), shard=shard).replace("world_size=2", "world_size=8")
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(8)]
    logs = [p.communicate(timeout=600)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    allx = np.concatenate(list(parts.values()))
    exp = orc.normalize_expected(orc.s2_expected_counts(allx, 18))
    for name, part in parts.items():
        ref = orc.s2_scores(part, 18, exp)
        with gzip.open(out / ("scores_in_s2_%s.txt.gz" % name), "rb") as gzf:
            text = gzf.read()
        starts = np.arange(part.shape[0]) * 200
        assert text == orc.format_scores_text(ref, name.split("_")[-1], starts, starts + 200)
    assert (out / "regionsOfInterest_in_s2.txt").exists() and not list(out.glob("temp_*"))
