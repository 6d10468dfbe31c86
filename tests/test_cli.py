"""`epilogos` command line mirror (epilogos_b200.run): flag validation on CPU, full local pipeline on the GPU."""
import gzip

import numpy as np
import pytest
from click.testing import CliRunner

from test_host_stages import write_tsv

META = "zero_index\tone_index\tshort_name\tlong_name\n" + "".join("%d\t%d\tS%d\tstate %d\n" % (i, i + 1, i + 1, i + 1)
                                                                      for i in range(18))


def test_flag_validation_messages(tmp_path):
    from epilogos_b200 import run
    r = CliRunner().invoke(run.main, ["-l", "-o", str(tmp_path), "-j", "x"])
    assert "ERROR: [-i, --input-directory] required in 'single' group mode" in r.output
    r = CliRunner().invoke(run.main, ["-m", "paired", "-a", str(tmp_path), "-o", str(tmp_path), "-j", "x"])
    assert "ERROR: [-b, --directory-two] required in 'paired' group mode" in r.output
    r = CliRunner().invoke(run.main, ["-i", str(tmp_path), "-o", str(tmp_path), "-j", "x", "-n"])
    assert "not compatible with [-n, --null-distribution]" in r.output
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    assert run.getNumStates(meta) == 18 and run.getStateNames(meta)[17] == "S18"
    inp = tmp_path / "in"
    inp.mkdir()
    (inp / "f.txt").write_text("chr1\t0\t200\t1\n")
    r = CliRunner().invoke(run.main, ["-i", str(inp), "-o", str(tmp_path / "o"), "-j", str(meta), "-s", "4"])
    assert isinstance(r.exception, ValueError) and "Saliency Metric Invalid" in str(r.exception)
    r = CliRunner().invoke(run.main, ["-i", str(tmp_path / "missing"), "-o", str(tmp_path / "o"), "-j", str(meta)])
    assert isinstance(r.exception, FileNotFoundError)
    r = CliRunner().invoke(run.main, ["-v"])
    assert "Version:" in r.output


@pytest.mark.gpu
def test_local_single_pipeline_end_to_end(tmp_path, golden):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import run, session
    from oracle import epilogos_oracle as orc, roi_oracle
    session.clear()
    g = golden("real10_chr1_k18")
    x = g["x"]
    inp = tmp_path / "mydata"; out = tmp_path / "out"
    inp.mkdir()
    write_tsv(inp / "epilogos_matrix_chr1.txt.gz", x, gz=True)
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    r = CliRunner().invoke(run.main, ["-l", "-i", str(inp), "-o", str(out), "-j", str(meta), "-s", "1", "-w", "20"])
    assert r.exit_code == 0, r.output + repr(r.exception)
    with gzip.open(out / "scores_mydata_s1_epilogos_matrix_chr1.txt.gz", "rb") as f:
        text = f.read()
    ref_lines = g["s1_text"].tobytes().split(b"\n")
    got_lines = text.split(b"\n")
    assert len(ref_lines) == len(got_lines) and sum(a != b for a, b in zip(ref_lines, got_lines)) <= 2
    # step 4 consumed the temp files and wrote the ROI list; compare with the oracle on the reference's scores
    assert not list(out.glob("temp_scores_*.npz")) and not (out / "exp_freq_mydata_s1.npy").exists()
    starts = np.arange(len(x), dtype=np.int64) * 200
    sel = roi_oracle.max_mean(starts, starts + 200, g["s1_scores"].sum(axis=1), 20, 100)
    states = roi_oracle.max_states(g["s1_scores"], sel["original_idx"], 20)
    want = roi_oracle.roi_text(np.array(["chr1"] * len(x), dtype=object), sel, states, ["S%d" % i for i in range(1, 19)])
    got = (out / "regionsOfInterest_mydata_s1.txt").read_text()
    assert [l.split("\t")[:4] for l in got.splitlines()] == [l.split("\t")[:4] for l in want.splitlines()]


def test_cli_main_end_to_end_on_cpu_with_the_oracle_backend(tmp_path, golden, monkeypatch):
    """The whole `epilogos -l` command path (argument checks, file discovery, prefetch, steps 1-4, clean-up) without a
    GPU: the session's backend is replaced by the oracle-backed stand-in of the host-stage tests, so this covers
    run.main / run.run_stages themselves; the GPU test above covers the same path with the CUDA backend."""
    from fake_backend import OracleBackend
    from epilogos_b200 import run, session
    from oracle import epilogos_oracle as orc
    session.clear()
    monkeypatch.setattr(session, "_backend", OracleBackend())
    x = golden("real10_chr1_k18")["x"][:1500]
    inp = tmp_path / "mydata"; out = tmp_path / "out"
    inp.mkdir()
    write_tsv(inp / "epilogos_matrix_chr1.txt.gz", x[:900], gz=True)
    write_tsv(inp / "epilogos_matrix_chr2.txt.gz", x[900:], chrom="chr2", gz=True)
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    r = CliRunner().invoke(run.main, ["-l", "-i", str(inp), "-o", str(out), "-j", str(meta), "-s", "2", "-w", "20"])
    assert r.exit_code == 0, r.output + repr(r.exception)
    assert "STEP 1" in r.output and "STEP 4" in r.output
    exp = orc.normalize_expected(orc.s2_expected_counts(x, 18))
    for name, part, chrom in (("chr1", x[:900], "chr1"), ("chr2", x[900:], "chr2")):
        with gzip.open(out / ("scores_mydata_s2_epilogos_matrix_%s.txt.gz" % name), "rb") as f:
            text = f.read()
        starts = np.arange(len(part)) * 200
        assert text == orc.format_scores_text(orc.s2_scores(part, 18, exp), chrom, starts, starts + 200)
    assert (out / "regionsOfInterest_mydata_s2.txt").exists()
    assert not list(out.glob("temp_*")) and not (out / "exp_freq_mydata_s2.npy").exists()
    session.clear()
    # the score -> ROI hand-over happened in memory (no temp_scores npz was ever written) and gives the very file that
    # the reference's route through temp_scores_*.npz gives (EPILOGOS_B200_KEEP_TEMP=1)
    assert not session.handover
    from epilogos_b200 import helpers
    written = []
    real = helpers.savez_level
    monkeypatch.setattr(helpers, "savez_level", lambda path, *a, **k: (written.append(str(path)), real(path, *a, **k))[1])
    out1 = tmp_path / "out_mem"
    r = CliRunner().invoke(run.main, ["-l", "-i", str(inp), "-o", str(out1), "-j", str(meta), "-s", "2", "-w", "20"])
    assert r.exit_code == 0 and not [w for w in written if "temp_scores" in w]
    monkeypatch.setenv("EPILOGOS_B200_KEEP_TEMP", "1")
    session.clear()
    out2 = tmp_path / "out_files"
    r = CliRunner().invoke(run.main, ["-l", "-i", str(inp), "-o", str(out2), "-j", str(meta), "-s", "2", "-w", "20"])
    assert r.exit_code == 0 and len([w for w in written if "temp_scores" in w]) == 2
    assert (out1 / "regionsOfInterest_mydata_s2.txt").read_text() == (out2 / "regionsOfInterest_mydata_s2.txt").read_text()
    assert (out / "regionsOfInterest_mydata_s2.txt").read_text() == (out2 / "regionsOfInterest_mydata_s2.txt").read_text()
    session.clear()


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference`: rank 0 prints ONE JSON line with the contract's keys (the unmodified reference staged under
    oracle/_ref or named by EPILOGOS_REFERENCE, else the oracle port), the same `config` object our arm prints, e2e = value;
    every other rank exits 0 without output."""
    import json
    import os
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    env = dict(os.environ, EPI_BENCH_REF_BUDGET_S="3")
    env.pop("RANK", None)
    r = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--config", "s2_genome_127"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "bins/s" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["e2e"] == {"value": d["value"], "unit": "bins/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["config"]["biosamples"] == 127 and d["config"]["states"] == 15 and "workload" in d["config"]
    r = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                       text=True, timeout=120, env=dict(env, RANK="1", WORLD_SIZE="2"))
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bench_dump_outputs_format(tmp_path):
    """bench.dump_outputs: float32 stays float32, integer tables become exact float64, a large table is written at a seeded
    sample of its entries, and the same call writes the same files."""
    import sys
    from pathlib import Path
    import torch
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    import bench
    rows = bench.sample_rows(5_000_000)
    assert len(rows) == bench.DUMP_ROWS and np.array_equal(rows, bench.sample_rows(5_000_000)) and (np.diff(rows) > 0).all()
    assert np.array_equal(bench.sample_rows(100), np.arange(100))
    scores = torch.arange(100 * 18, dtype=torch.float32).reshape(100, 18)
    table = torch.arange(18 * 18, dtype=torch.int64).reshape(18, 18) + (1 << 40)
    big = torch.arange(bench.DUMP_ENTRIES + 5, dtype=torch.float32)
    wide = torch.arange((bench.DUMP_ENTRIES // 18 + 1) * 18, dtype=torch.float32).reshape(-1, 18)   # per-bin: written whole
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(d, np.array([3, 50]), {"scores": bench.take_rows(scores, np.array([3, 50])), "wide": wide},
                           {"expected_counts": table, "big": big})
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["big.npy", "big_entries.npy", "expected_counts.npy", "rows.npy", "scores.npy", "wide.npy"]
    for n in names:
        assert (tmp_path / "a" / n).read_bytes() == (tmp_path / "b" / n).read_bytes()
    s = np.load(tmp_path / "a" / "scores.npy")
    assert s.dtype == np.float32 and np.array_equal(s, scores.numpy()[[3, 50]])
    t = np.load(tmp_path / "a" / "expected_counts.npy")
    assert t.dtype == np.float64 and np.array_equal(t.astype(np.int64), table.numpy())
    b, e = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "a" / "big_entries.npy")
    assert b.shape == (bench.DUMP_ENTRIES,) and np.array_equal(b, e.astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "a" / "wide.npy"), wide.numpy())


@pytest.mark.gpu
def test_bench_dump_outputs_repeat(tmp_path):
    """`bench.py --dump-outputs`: two runs with the same arguments write the same outputs, and the dumped table has its
    closed form (S2 counts sum to bins C (C-1))."""
    import json
    import os
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    env = dict(os.environ, EPI_BENCH_NO_CLOCKS="1")
    for run_dir in ("a", "b"):
        r = subprocess.run([sys.executable, str(root / "bench.py"), "--steps", "2", "--warmup", "0", "--bins", "300000",
                            "--no-e2e", "--no-target", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run_dir)],
                           capture_output=True, text=True, timeout=600, env=env)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 2 and line["check"] == "ok"
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["expected.npy", "expected_counts.npy", "rows.npy", "scores.npy"]
    for n in names:
        assert np.array_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n))
    counts = np.load(tmp_path / "a" / "expected_counts.npy")
    scores = np.load(tmp_path / "a" / "scores.npy")
    assert counts.shape == (18, 18) and counts.sum() == 300000 * 833 * 832
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.shape == (1 << 18,) and rows.max() < 300000 and scores.shape == (1 << 18, 18)
    assert scores.dtype == np.float32 and np.isfinite(scores).all()


# per configuration: the engine call made once per step, and the passes outside the timed loop (S2: 3 warm-up passes at
# --warmup 0 and 3 more after the clock sampler starts; S3 and paired: 1 warm-up pass; paired: 1 untimed pass for the dump)
STEP_CALLS = {"s2_genome_833": ("bin_counts", 6), "s3_chr1_833": ("s3_expected_tiles", 1), "paired_s1_chr1": ("quiescent_mask", 2)}
DUMP_FILES = {"s2_genome_833": {"expected", "expected_counts", "rows", "scores"},
              "s3_chr1_833": {"expected", "expected_entries", "rows", "scores"},
              "paired_s1_chr1": {"delta", "distance", "expected", "max_diff_state", "null_distances", "quiescent", "rows"}}


@pytest.mark.gpu
@pytest.mark.parametrize("config", sorted(STEP_CALLS))
def test_bench_steps_and_dump_per_config(tmp_path, monkeypatch, capsys, config):
    """In process, so the engine's calls can be counted: `--steps 4` runs exactly 4 timed steps in every configuration (S3
    and paired mode used to stop at 3), and each configuration's dump holds its outputs at the documented sizes."""
    import json
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    import bench
    from epilogos_b200 import engine
    name, outside = STEP_CALLS[config]
    calls = []
    real = getattr(engine, name)
    monkeypatch.setattr(engine, name, lambda *a, **k: (calls.append(1), real(*a, **k))[1])
    monkeypatch.setenv("EPI_BENCH_NO_CLOCKS", "1")
    steps, bins = 4, 20000
    monkeypatch.setattr(sys, "argv", ["bench.py", "--config", config, "--steps", str(steps), "--warmup", "0", "--bins",
                                      str(bins), "--no-e2e", "--no-target", "--no-cpu-baseline", "--dump-outputs",
                                      str(tmp_path)])
    bench.main()
    line = json.loads([ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == steps and len(calls) == steps + outside
    out = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert set(out) == DUMP_FILES[config]
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    if config == "s3_chr1_833":
        assert out["scores"].shape == (bins, 18) and np.array_equal(out["rows"], np.arange(bins))
        assert out["expected"].shape == out["expected_entries"].shape == (bench.DUMP_ENTRIES,)
        assert out["expected_entries"].max() < 833 * 833 * 18 * 18
    if config == "paired_s1_chr1":
        n = bench.DUMP_ROWS // 64
        assert out["rows"].shape == (n,) and out["delta"].shape == (n, 18) and out["null_distances"].shape == (n, 1000)
        assert out["expected"].shape == (18,) and abs(float(out["expected"].sum()) - 1.0) < 1e-5
