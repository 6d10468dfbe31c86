#!/usr/bin/env python
"""bench.py -- bins/sec for expected + scores on B200 (BASELINE.json metric), plus the CPU reference arm.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config ...] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one synthetic matrix that is already resident in HBM:
K1 counts -> K2 expected table (tensor-core Gram of the count bytes) -> (allreduce over ranks) -> K4 normalise ->
K5 scores (S2: table preparation + tensor-core mat-vec kernel + the gated DIRECT fallback = 6 launches per step).
Workload of `value` at every N: BASELINE.json configs[1], S2 on 15.5 M bins x 833 biosamples x 18 states PER GPU
(weak scaling; the bins shard with no data-path collective, only the 18x18 table is all-reduced).
The matrix (13 GB) is far larger than L2 (126 MB), so no L2 flush is needed between steps.

Beside it, in the same JSON line:
  check         the all-reduced integer table equals its closed form on every rank (correctness travels with the number)
  target        the north-star configuration: ONE genome sharded over the N GPUs (strong scaling) for S2 and S1, eager and
                as a captured CUDA graph, and ONE chr1 for S3 with Gram / tile all-reduce / scores timed separately
  e2e           the same metric through the reference-facing C-ABI calls with pinned HOST buffers, H2D and D2H inside the
                timed region (epi_single_host_packed: the matrix in the 4/5-bit packed transport layout; the int8 variant
                beside it; S3 and paired configurations through epi_s3_host / epi_paired_host)
  cpu_baseline  N = 1 only: the UNMODIFIED reference (oracle/_ref, byte-compiled by __graft_entry__.build()) on the box's host cores

`--dump-outputs DIR` writes what our arm's timed path computed in its last step as DIR/<name>.npy (dump_outputs below): the
inputs are seeded, so two builds run with the same arguments can be compared output for output.

`--impl reference` times that reference -- expected.main -> expectedCombination.main -> scores.main with one worker
process per core on a bounded TSV.gz sample of the workload, parse and gz write included (kind "reference"; the oracle's
row-loop port is the fallback when nothing was staged).
"""
import argparse
import json
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

GENOME_BINS = 15_500_000
CONFIGS = {
    # name: (bins per GPU, biosamples, states, description)
    "s2_genome_833": (GENOME_BINS, 833, 18, "S2 whole-genome 15.5M bins x 833 biosamples, 18-state (BASELINE configs[1])"),
    "s2_genome_127": (GENOME_BINS, 127, 15, "S2 whole-genome 15.5M bins x 127 biosamples, 15-state (BASELINE configs[4])"),
    "s1_chr1_833": (1_246_253, 833, 18, "S1 chr1 1,246,253 bins x 833 biosamples, 18-state (shape of BASELINE configs[0])"),
    "s3_chr1_833": (1_250_000, 833, 18, "S3 chr1 1.25M bins x 833 biosamples, 18-state (BASELINE configs[2])"),
    "paired_s1_chr1": (1_250_000, 833, 18, "paired S1 chr1 1.25M bins, groups of 400 + 433 biosamples, 18-state, 1000 null "
                                            "permutations per bin (BASELINE configs[3])"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps; with --impl reference each is one full pass of the reference (for S3 tens of "
                         "seconds of set-up each, which the sample budget does not bound)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="s2_genome_833", choices=sorted(CONFIGS))
    ap.add_argument("--bins", type=int, default=0, help="override bins per GPU (debug)")
    ap.add_argument("--kind", default="realistic", choices=["realistic", "uniform"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-target", action="store_true", help="skip the strong-scaling target sections (S2 / S1 genome, S3 chr1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (our arm only; with several GPUs, "
                         "the tables and rank 0's bins)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


DUMP_SEED = 20261020
DUMP_ROWS = 1 << 18                 # bins written from a longer per-bin output (19 MB of float32 scores at 18 states)
DUMP_ENTRIES = 1 << 20              # entries written from a larger table (the S3 table holds C*C*K*K)


def sample_rows(bins, n=DUMP_ROWS):
    """A fixed, seeded, sorted sample of n of the bins (all bins when there are no more than n)."""
    import numpy as np
    if bins <= n:
        return np.arange(bins)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(bins, n, replace=False))


def take_rows(t, rows):
    """Rows `rows` of the device tensor t (per-bin output, bins on dimension 0)."""
    import torch
    return t.index_select(0, torch.from_numpy(rows).to(t.device))


def dump_outputs(directory, rows, per_bin, tables):
    """--dump-outputs: every array as DIR/<name>.npy, float32 kept as float32 and every other type as float64 (exact for the
    integer tables), with the sampled bin indices as rows.npy.  `per_bin` arrays arrive already taken at `rows` and are
    written whole; a table of more than DUMP_ENTRIES entries is written at a fixed, seeded sample of its flat entries,
    indices in <name>_entries.npy.  Everything stays within 64 MB."""
    import numpy as np
    d = Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    out = {"rows": rows}
    out.update({name: t.cpu().numpy() for name, t in per_bin.items()})
    for name, t in tables.items():
        a = t.cpu().numpy()
        if a.size > DUMP_ENTRIES:
            pick = np.sort(np.random.default_rng(DUMP_SEED).choice(a.size, DUMP_ENTRIES, replace=False))
            out[name + "_entries"] = pick
            a = a.reshape(-1)[pick]
        out[name] = a
    out = {name: a.astype(np.float32 if a.dtype == np.float32 else np.float64) for name, a in out.items()}
    total = sum(a.nbytes for a in out.values())
    if total > 64 << 20:
        raise RuntimeError("--dump-outputs: %d bytes exceed 64 MB" % total)
    for name, a in out.items():
        np.save(d / (name + ".npy"), a)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm.  kind "reference": the UNMODIFIED reference (oracle/_ref, byte-compiled by oracle/stage_reference.py from the
# checkout EPILOGOS_REFERENCE names) runs its own expected.main -> expectedCombination.main -> scores.main on a TSV.gz
# sample of the workload with one worker process per host core -- what `epilogos -l -c 0` executes before the ROI step
# (run.py:191-279), TSV parse and gz write included; its own verbose timers give the compute-only share.  kind "port": the oracle's
# row-loop port (same algorithm and cost, I/O excluded), the fallback when the reference was not staged.
# ------------------------------------------------------------------------------------------------
def config_dict(args, world, bins, cols, k, desc, pitch=None):
    """The `config` object of the JSON line: identical for our arm and the reference arm."""
    saliency = 1 if args.config.startswith("paired") else int(args.config[1])
    return {"workload": desc, "bins_per_gpu": bins, "biosamples": cols, "states": k, "saliency": saliency,
            "distribution": args.kind,
            "parallelism": "bins sharded x%d, integer table allreduce" % world,
            "l2": "inputs (%.1f GB/GPU) larger than L2, no flush needed" % (bins * (pitch or ((cols + 15) & ~15)) / 1e9)}


def _reference_staged():
    try:
        from oracle import stage_reference
        return stage_reference.staged_root() is not None
    except Exception:
        return False


def _write_sample(path, states0):
    """One input matrix of the sample as TSV.gz (README.md:286-292), outside every timed region.  Inside our own arm (the
    `cpu_baseline` leg, where the library is loaded anyway) the library's native writer; in the `--impl reference` process
    nothing of this repository's engine is loaded, so the oracle's vectorised Python writer (~10 s per 100,000 x 833 rows).
    Same text either way."""
    if "epilogos_b200._lib" in sys.modules:
        try:
            from epilogos_b200 import preprocess
            preprocess.write_matrix(path, "chr1", states0, gzip_level=1)
            return
        except Exception:
            pass
    from oracle import reference_driver as ref
    ref.write_matrix_tsv_gz(path, states0)


def _sample_files(workdir, config, bins, cols, k, kind, seed=4242):
    """Write the TSV.gz sample of `bins` rows of the configuration; returns (file1, file2)."""
    from oracle import epilogos_oracle as orc
    workdir = Path(workdir)
    if config.startswith("paired"):
        a, b = workdir / "A", workdir / "B"
        a.mkdir(exist_ok=True)
        b.mkdir(exist_ok=True)
        _write_sample(a / "epilogos_matrix_chr1.txt.gz", orc.synth_states(bins, 400, k, seed, kind))
        _write_sample(b / "epilogos_matrix_chr1.txt.gz", orc.synth_states(bins, 433, k, seed + 1, kind))
        return a / "epilogos_matrix_chr1.txt.gz", b / "epilogos_matrix_chr1.txt.gz"
    d = workdir / "in"
    d.mkdir(exist_ok=True)
    f = d / "epilogos_matrix_chr1.txt.gz"
    _write_sample(f, orc.synth_states(bins, cols, k, seed, kind))
    return f, "null"


def _s3_workers(cores, cols, k):
    """scores.s3Score needs ~6 x the float32 [C,C,K,K] table per worker (masked temporaries of klScoreND, scores.py:479-480)
    and expected.s3Calc pickles one int32 table per worker back: cap the pool by the memory that is available."""
    table = cols * cols * k * k * 4
    avail = 64 << 30
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                avail = int(line.split()[1]) * 1024
    except OSError:
        pass
    return max(1, min(cores, int(avail * 0.6 // (7 * table + (1 << 30)))))


def reference_cpu_arm(args, steps, warmup, budget_s):
    """Times the staged reference on bounded samples.  Returns (dict cpu_baseline, list of per-step seconds, bins per step)."""
    import tempfile
    from oracle import reference_driver as ref
    bins_full, cols, k, _ = CONFIGS[args.config]
    paired = args.config.startswith("paired")
    saliency = 1 if paired else int(args.config[1])
    cores = os.cpu_count() or 1
    nproc = _s3_workers(cores, cols, k) if saliency == 3 else cores
    per_step = max(2.0, min(20.0, budget_s / max(1, steps + warmup)))
    unit = 2 if saliency == 3 else 64                  # rows per worker in the smallest probe
    with tempfile.TemporaryDirectory(prefix="epi_ref_") as d:
        # two-point calibration t(n) = a + b n on warm imports (a = pool start-up, table load / store, first-row parse)
        n1, n2 = nproc * unit, nproc * unit * 4
        probe = []
        for n in (n1, n1, n2):                         # the first run also pays the imports: dropped
            f1, f2 = _sample_files(d, args.config, n, cols, k, args.kind)
            probe.append(ref.time_pipeline(f1, f2, k, saliency, nproc, d)[0])
        t1, t2 = probe[1], probe[2]
        b = max((t2 - t1) / (n2 - n1), 1e-7)
        a = max(t1 - b * n1, 0.0)
        n = int(max(n2, min(bins_full, 400_000, (per_step - a) / b)))
        if saliency == 3:           # the fixed set-up (tens of seconds) would leave no rows at all: time at least 32 rows per worker
            n = max(n, nproc * 32)
        n = max(nproc, n // nproc * nproc)
        f1, f2 = _sample_files(d, args.config, n, cols, k, args.kind)
        times, compute = [], []
        for it in range(warmup + steps):
            wall, comp = ref.time_pipeline(f1, f2, k, saliency, nproc, d, verbose_timers=(it == warmup + steps - 1))
            if it >= warmup:
                times.append(wall)
            if comp:
                compute.append(comp)
    sec = sum(times) / len(times)
    what = "paired S1 (groups of 400 + 433 biosamples, one null shuffle per bin)" if paired else "S%d" % saliency
    base = dict(value=n / sec, unit="bins/s", cores=nproc, kind="reference",
                sample="%d bins x %d biosamples x %d states as TSV.gz, %s: the unmodified reference's expected.main -> "
                       "expectedCombination.main -> scores.main with %d worker processes (what `epilogos -l` runs before the "
                       "ROI step), TSV parse and scores gz write included; %.2f s per pass, fixed cost %.2f s"
                       % (n, cols, k, what, nproc, sec, a),
                host_cores=cores)
    if compute:
        # the last pass ran with the reference's verbose timers on: compute loops of the first worker (all workers get
        # equal row ranges and run concurrently), I/O and process start-up excluded
        base["compute_only"] = {"value": n / compute[-1], "unit": "bins/s",
                                "how": "reference's own verbose timers (expected.py:114,160,202; scores.py:324,423,506), "
                                       "first worker, last pass"}
    return base, times, n


def _cpu_worker(args):
    from oracle import epilogos_oracle as orc
    bins, cols, k, saliency, seed, phase, exp = args
    x = orc.synth_states(bins, cols, k, seed)
    if phase == "expected":
        if saliency == 1:
            return orc.s1_expected_counts_rowloop(x, k)
        return orc.s2_expected_counts_rowloop(x, k)
    if saliency == 1:
        return orc.s1_scores_rowloop(x, k, exp).sum()
    return orc.s2_scores_rowloop(x, k, exp).sum()


def cpu_port_pass(pool, cores, bins_per_core, cols, k, saliency, seed0):
    """expected.main -> expectedCombination.main -> scores.main on cores*bins_per_core bins, one row range
    per worker process (the reference's multiprocessing.Pool fan-out, expected.py:71-79, scores.py:147-154).
    Returns seconds spent in the two compute phases (synthetic chunk generation included in the workers is
    measured separately and subtracted)."""
    from oracle import epilogos_oracle as orc
    jobs = [(bins_per_core, cols, k, saliency, seed0 + i, "expected", None) for i in range(cores)]
    t0 = time.perf_counter()
    parts = pool.map(_cpu_worker, jobs)
    exp = orc.normalize_expected(sum(parts))
    jobs = [(bins_per_core, cols, k, saliency, seed0 + i, "scores", exp) for i in range(cores)]
    pool.map(_cpu_worker, jobs)
    return time.perf_counter() - t0


def _gen_worker(args):
    from oracle import epilogos_oracle as orc
    bins, cols, k, seed = args
    return int(orc.synth_states(bins, cols, k, seed).sum())


def port_cpu_arm(cols, k, saliency, steps, warmup, budget_s):
    """Fallback when the reference is not staged: the oracle's row-loop port, S1 / S2 only."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    ctx = mp.get_context("fork")
    per_step = max(2.0, min(20.0, budget_s / max(1, steps + warmup)))
    with ctx.Pool(cores) as pool:
        cpu_port_pass(pool, cores, 64, cols, k, saliency, 900)                 # warm pool and imports
        t1 = cpu_port_pass(pool, cores, 256, cols, k, saliency, 1000)
        t2 = cpu_port_pass(pool, cores, 1024, cols, k, saliency, 1100)
        b = max((t2 - t1) / 768.0, 1e-7)
        per_core = int(max(256, min(50000, (per_step - max(t1 - 256 * b, 0.0)) / b)))
        times = []
        for it in range(warmup + steps):
            tt = cpu_port_pass(pool, cores, per_core, cols, k, saliency, 2000 + 100 * it)
            tg0 = time.perf_counter()
            pool.map(_gen_worker, [(per_core, cols, k, 2000 + 100 * it + i) for i in range(cores)])
            tgen = 2 * (time.perf_counter() - tg0)
            if it >= warmup:
                times.append(max(tt - tgen, 1e-6))
    total = per_core * cores
    sec = sum(times) / len(times)
    return dict(value=total / sec, unit="bins/s", cores=cores, kind="port",
                sample="%d bins x %d biosamples x %d states (S%d expected+scores, %d worker processes x %d bins, "
                       "row-loop port of expected.py/scores.py, I/O excluded)" % (total, cols, k, saliency, cores,
                                                                                  per_core)), times, total


def cpu_arm(args, steps, warmup, budget_s):
    if _reference_staged():
        return reference_cpu_arm(args, steps, warmup, budget_s)
    _, cols, k, _ = CONFIGS[args.config]
    if args.config.startswith("paired") or args.config[1] == "3":
        raise RuntimeError("the reference was not built into oracle/_ref and the port covers S1/S2 only")
    return port_cpu_arm(cols, k, int(args.config[1]), steps, warmup, budget_s)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    bins, cols, k, desc = CONFIGS[args.config]
    paired = args.config.startswith("paired")
    saliency = 1 if paired else int(args.config[1])
    steps, warmup = args.steps, args.warmup
    if saliency == 3:               # one pass costs tens of seconds of fixed set-up per worker (693k-tuple pair list, 0.9 GB tables)
        warmup = 0
    base, times, n = cpu_arm(args, steps, warmup, budget_s=float(os.environ.get("EPI_BENCH_REF_BUDGET_S", "150")))
    sec = sum(times) / len(times)
    metric = ("bins/sec for paired expected+scores (S1)" if paired else "bins/sec for expected+scores (S%d)" % saliency)
    line = {
        "impl": "reference", "metric": metric, "value": base["value"],
        "unit": "bins/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64+f64" if saliency != 3 else "int32+f32 (the reference's S3 arithmetic)", "data": "synthetic",
        "config": config_dict(args, max(1, args.gpus), bins, cols, k, desc),
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "bins/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "bins_per_step": n,
        "note": "each step is one pass of the reference over a bounded sample of the workload on the host CPU",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampling through NVML while the timed region runs
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / throttle reasons of one GPU while the timed region runs, taken by a SEPARATE `nvidia-smi -lms` process
    (the recipe's clocks line).  An in-process NVML poller was measured to cost 0.25 ms per 3 ms step at 2 GPUs: its
    driver calls serialise with rank 0's kernel launches and the other rank then waits at the all-reduce."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap,clocks_event_reasons.hw_power_brake_slowdown")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap", "hw_power_brake_slowdown"]

    def __init__(self, index):
        import subprocess
        import tempfile
        self.t_lo = self.t_hi = None
        self.out = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        period = os.environ.get("EPI_BENCH_CLOCK_PERIOD_MS", "20")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", period],
                                         stdout=self.out, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def start(self):
        """Call right before the timed region (the process is already sampling)."""
        self.t_lo = time.time()

    def stop(self):
        self.t_hi = time.time()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "power_w_max": None}
        time.sleep(0.03)                     # let the sample that straddles the end land
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.flush()
        self.out.seek(0)
        import datetime
        rows = []
        for line in self.out.read().splitlines():
            f = [v.strip() for v in line.split(",")]
            if len(f) != 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, int(float(f[1])), int(float(f[2])), float(f[3]), [x.lower().startswith("active") for x in f[4:]]))
            except ValueError:
                continue
        self.out.close()
        try:
            os.unlink(self.out.name)
        except OSError:
            pass
        inside = [r for r in rows if self.t_lo - 0.005 <= r[0] <= self.t_hi + 0.005]
        if not inside and rows:              # region shorter than the sampling period: take the nearest sample
            mid = 0.5 * (self.t_lo + self.t_hi)
            inside = [min(rows, key=lambda r: abs(r[0] - mid))]
        clk = sorted(r[1] for r in inside)
        reasons = sorted({n for r in inside for n, on in zip(self.NAMES, r[4]) if on})
        return {"sm_mhz": clk[len(clk) // 2] if clk else None, "sm_max_mhz": inside[0][2] if inside else None,
                "reasons": reasons, "samples": len(inside), "power_w_max": max((r[3] for r in inside), default=None),
                "how": "nvidia-smi -lms %s in a separate process, samples inside the timed region" %
                       os.environ.get("EPI_BENCH_CLOCK_PERIOD_MS", "20")}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def _timed_loop(torch, dist, world, stream, fn, steps):
    """barrier + synchronize, `steps` calls of fn() between two CUDA events on the launching stream, synchronize + barrier;
    returns ms per step, MAX over the ranks."""
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(steps):
        fn()
    t1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([t0.elapsed_time(t1) / steps], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def _make_step(torch, dist, engine, world, x, cols, k, saliency, cnt, scores):
    """One pass of the S1/S2 hot path over the resident matrix x; returns (step function, dict with the last tables)."""
    last = {}

    def step():
        engine.bin_counts(x, cols, k, out=cnt)                                                      # K1
        n1, n2 = engine.expected_tables(cnt, cols, want_s1=saliency == 1, want_s2=saliency == 2)    # K2
        n = n1 if saliency == 1 else n2
        if world > 1 and not os.environ.get("EPI_BENCH_SKIP_ALLREDUCE"):
            dist.all_reduce(n)                                                                      # the path's only exchange
        e = engine.normalize(n)                                                                     # K4
        if saliency == 1:
            engine.scores_s1(cnt, cols, e, out32=scores)                                            # K5
        else:
            engine.scores_s2(cnt, cols, e, out32=scores)
        last["n"], last["e"] = n, e
    return step, last


def _check_step(torch, dist, world, last, total_bins, cols, saliency, scores):
    """Correctness carried by the benchmark line itself: the all-reduced integer table must sum to its closed form
    (S1: bins C, S2: bins C (C-1); SURVEY 8a) on every rank, every rank must hold the same table, and the scores are finite."""
    want = total_bins * cols * (cols - 1 if saliency == 2 else 1)
    got = int(last["n"].sum().item())
    ok = got == want and bool(torch.isfinite(scores[:: max(1, scores.shape[0] // 65536)]).all())
    if world > 1:
        ref = last["n"].clone()
        dist.broadcast(ref, src=0)
        ok = ok and bool(torch.equal(ref, last["n"]))
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    return "ok" if ok else "FAILED: table sum %d, closed form %d" % (got, want), want


def _strong_section(torch, dist, engine, world, x, cols, k, saliency, total_bins, steps):
    """The north-star target configuration: ONE whole genome (total_bins) sharded over the `world` GPUs (strong scaling).
    Every rank runs the step on total_bins / world rows; timed eagerly and as a captured CUDA graph (at 1/8 of a genome the
    step is ~0.4 ms and the ~8 launches + the all-reduce are a visible fixed cost)."""
    stream = torch.cuda.current_stream()
    lo, hi = total_bins * int(os.environ.get("RANK", "0")) // world, total_bins * (int(os.environ.get("RANK", "0")) + 1) // world
    rows = hi - lo
    xs = x[:rows]
    cnt = torch.empty((rows, k), dtype=torch.int16, device="cuda")
    scores = torch.empty((rows, k), dtype=torch.float32, device="cuda")
    step, last = _make_step(torch, dist, engine, world, xs, cols, k, saliency, cnt, scores)
    for _ in range(3):
        step()
    eager_ms = _timed_loop(torch, dist, world, stream, step, steps)
    check, _ = _check_step(torch, dist, world, last, total_bins, cols, saliency, scores)
    out = {"bins_total": total_bins, "bins_per_gpu": rows, "saliency": saliency, "ms_per_step_eager": eager_ms,
           "value_eager": total_bins / (eager_ms * 1e-3), "check": check}
    graph_ms = None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(stream)
        with torch.cuda.stream(side):
            step()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                step()
        stream.wait_stream(side)
        torch.cuda.synchronize()
        for _ in range(3):
            g.replay()
        graph_ms = _timed_loop(torch, dist, world, stream, g.replay, steps)
        check_g, _ = _check_step(torch, dist, world, last, total_bins, cols, saliency, scores)
        out.update({"ms_per_step_graph": graph_ms, "value_graph": total_bins / (graph_ms * 1e-3), "check_graph": check_g})
        del g
    except Exception as exc:                       # capture is an optimisation: report why it was not available
        out["graph_error"] = str(exc)[:200]
        torch.cuda.synchronize()
    best = min(eager_ms, graph_ms) if graph_ms else eager_ms
    out.update({"ms_per_step": best, "value": total_bins / (best * 1e-3), "unit": "bins/s", "scaling": "strong"})
    return out


def _s3_strong_section(torch, dist, engine, synth, world, rank, total_bins, cols, k, steps=2):
    """BASELINE configs[2] sharded over the GPUs: chr1 (1.25 M bins) split in `world` row ranges; every rank builds the
    tiles of its rows' one-hot Gram matrix, the ranks all-reduce the 464 MB int32 tile buffer (timed separately), every
    rank finalises the table and scores its own rows."""
    stream = torch.cuda.current_stream()
    lo, hi = total_bins * rank // world, total_bins * (rank + 1) // world
    rows = hi - lo
    x = synth.synth_states_device(rows, cols, k, seed=4321 + rank)
    plan = engine.s3_plan(rows, cols, k)
    tiles = torch.empty(plan["tile_bytes"] // 4, dtype=torch.int32, device="cuda")
    scores = torch.empty((rows, k), dtype=torch.float32, device="cuda")
    ev = {"gram": [], "allreduce": [], "score": []}
    keep = {}

    def step():
        e = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        e[0].record(stream)
        engine.s3_expected_tiles(x, cols, k, tiles=tiles)
        e[1].record(stream)
        if world > 1:
            dist.all_reduce(tiles[: plan["ntiles"] * 128 * 256])
        e[2].record(stream)
        counts, exp3 = engine.s3_finalize(tiles, cols, k, plan["mp"], total_bins, want_counts=False, want_exp=True)
        terms = engine.s3_terms(exp3.reshape(-1), cols, k)
        e[3].record(stream)
        engine.scores_s3(x, cols, k, terms, out32=scores)
        e[4].record(stream)
        ev["gram"].append((e[0], e[1]))
        ev["allreduce"].append((e[1], e[2]))
        ev["score"].append((e[3], e[4]))
        keep["exp3"] = exp3
    step()
    for v in ev.values():
        v.clear()
    ms = _timed_loop(torch, dist, world, stream, step, steps)
    parts = torch.tensor([sum(a.elapsed_time(b) for a, b in ev[n]) / len(ev[n]) for n in ("gram", "allreduce", "score")],
                         device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(parts, op=dist.ReduceOp.MAX)
    # closed form: the float32 table sums to 1 and the tile buffer's off-diagonal-block entries to bins C (C-1)
    total = float(keep["exp3"].double().sum().item())
    ck = cols * k
    useful = total_bins * ck * (ck + 1)
    return {"bins_total": total_bins, "bins_per_gpu": rows, "saliency": 3, "ms_per_step": ms,
            "value": total_bins / (ms * 1e-3), "unit": "bins/s", "scaling": "strong",
            "gram_ms": float(parts[0]), "allreduce_ms": float(parts[1]), "score_ms": float(parts[2]),
            "allreduce_bytes": int(plan["ntiles"]) * 128 * 256 * 4,
            "gram_useful_TOPS": useful / world / (float(parts[0]) * 1e-3) / 1e12,
            "check": "ok" if abs(total - 1.0) < 1e-5 else "FAILED: expected table sums to %r" % total}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from epilogos_b200 import engine, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        from epilogos_b200 import dist as edist
        edist.bind_to_gpu_numa(local)          # pinned host buffers and copies on the GPU's own socket
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    bins, cols, k, desc = CONFIGS[args.config]
    if args.bins:
        bins = args.bins
    engine.device_info()
    if args.config.startswith("paired"):
        return run_ours_paired(args, engine, synth, dist, world, rank, local, bins, cols, k, desc)
    saliency = int(args.config[1])
    if saliency == 3:
        return run_ours_s3(args, engine, synth, dist, world, rank, local, bins, cols, k, desc)

    x = synth.synth_states_device(bins, cols, k, seed=1234 + rank, kind=args.kind)
    cnt = torch.empty((bins, k), dtype=torch.int16, device="cuda")
    scores = torch.empty((bins, k), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream()
    k1_ev = []
    plain_step, last = _make_step(torch, dist, engine, world, x, cols, k, saliency, cnt, scores)

    def step(timed):
        if not timed:
            return plain_step()
        # same launches, with a pair of events around K1 (the kernel of the `roofline` object)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        engine.bin_counts(x, cols, k, out=cnt)
        e1.record(stream)
        k1_ev.append((e0, e1))
        n1, n2 = engine.expected_tables(cnt, cols, want_s1=saliency == 1, want_s2=saliency == 2)
        n = n1 if saliency == 1 else n2
        if world > 1 and not os.environ.get("EPI_BENCH_SKIP_ALLREDUCE"):
            dist.all_reduce(n)
        e = engine.normalize(n)
        if saliency == 1:
            engine.scores_s1(cnt, cols, e, out32=scores)
        else:
            engine.scores_s2(cnt, cols, e, out32=scores)
        last["n"], last["e"] = n, e

    sampler = ClockSampler(local) if rank == 0 and not os.environ.get("EPI_BENCH_NO_CLOCKS") else None
    for _ in range(max(3, args.warmup)):
        step(False)
    torch.cuda.synchronize()
    if rank == 0:
        time.sleep(0.3)                      # nvidia-smi needs a moment to start sampling
    if world > 1:
        dist.barrier()
    for _ in range(3):                       # every rank: back under load after the pause (collectives stay matched)
        step(False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if sampler:
        sampler.start()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(args.steps):
        step(not os.environ.get("EPI_BENCH_NO_K1_EVENTS"))
    t1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if sampler else None
    elapsed_ms = torch.tensor([t0.elapsed_time(t1)], device="cuda", dtype=torch.float64)
    k1_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in k1_ev) / max(1, len(k1_ev)) if k1_ev else 1.0], device="cuda",
                         dtype=torch.float64)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(k1_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(elapsed_ms.item()) / args.steps
    value = bins * world / (ms_per_step * 1e-3)
    k1_ms = float(k1_ms.item())
    check, _ = _check_step(torch, dist, world, last, bins * world, cols, saliency, scores)
    if args.dump_outputs and rank == 0:
        rows = sample_rows(bins)
        dump_outputs(args.dump_outputs, rows, {"scores": take_rows(scores, rows)},
                     {"expected_counts": last["n"], "expected": last["e"]})

    # ---- the north-star target: ONE genome / ONE chr1 sharded over the GPUs (strong scaling), S2, S1 and S3 ----
    target = None
    if args.config == "s2_genome_833" and not args.no_target and not args.bins:
        target = {}
        for name, fn in (("s2", lambda: _strong_section(torch, dist, engine, world, x, cols, k, 2, GENOME_BINS, args.steps)),
                         ("s1", lambda: _strong_section(torch, dist, engine, world, x, cols, k, 1, GENOME_BINS, args.steps)),
                         ("s3_chr1", lambda: _s3_strong_section(torch, dist, engine, synth, world, rank, 1_250_000, cols, k))):
            try:
                target[name] = fn()
            except Exception as exc:
                target[name] = {"error": str(exc)[:300]}
                torch.cuda.synchronize()
            torch.cuda.empty_cache()

    # ---- end to end through the host-buffer C-ABI call ----
    e2e = None
    if not args.no_e2e:
        e2e = _e2e_section(torch, dist, engine, world, x, bins, cols, k, saliency, args.e2e_steps)

    if rank == 0:
        peak, peak_src = peaks()
        achieved = bins * cols / (k1_ms * 1e-3) / 1e9
        traffic = None
        tf = ROOT / "profiles" / "roofline_traffic.json"
        if tf.exists():
            try:
                per_bin = json.loads(tf.read_text()).get(args.config, {}).get("k1_dram_bytes_per_bin")
                traffic = per_bin * bins if per_bin else None
            except Exception:
                traffic = None
        step_alg = bins * (cols + 4 * k)
        line = {
            "metric": "bins/sec for expected+scores (S%d)" % saliency, "value": value, "unit": "bins/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64",
            "data": "synthetic", "check": check,
            "config": config_dict(args, world, bins, cols, k, desc, pitch=int(x.shape[1])),
            "roofline": {"bound": "hbm", "kernel": "k1_counts_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bins * cols, "ms_per_launch": k1_ms},
            "step_roofline": {"algorithmic_bytes_per_step": step_alg, "achieved": step_alg / (ms_per_step * 1e-3) / 1e9,
                              "frac": step_alg / (ms_per_step * 1e-3) / 1e9 / peak, "unit": "GB/s"},
            "e2e": e2e, "gpu_launches": LAUNCHES_PER_STEP[saliency] * args.steps, "clocks": clocks,
        }
        if target is not None:
            line["target"] = target
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_arm(args, 1, 0, budget_s=12.0)[0]
            except Exception as exc:
                line["cpu_baseline"] = {"error": str(exc)[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# our kernels launched per step: K1, K2, K4, then S2: table preparation + tensor-core scores + gated DIRECT fallback;
# S1: value table + look-up kernel
LAUNCHES_PER_STEP = {1: 5, 2: 6}


def _e2e_section(torch, dist, engine, world, x, bins, cols, k, saliency, steps):
    """The same metric through the reference-facing C-ABI calls with the matrix in pinned HOST memory: H2D of the matrix and
    D2H of tables + scores are inside the timed region.  Headline: epi_single_host_packed -- the host buffer is the
    bit-packed transport layout the packer produces (5 bits per label for 18 states, 4 for <= 16), expanded on the device;
    `int8_layout` is epi_single_host on the plain int8 matrix of the same rows."""
    def timed(fn):
        fn()                                                                 # warm-up (allocations)
        if world > 1:
            dist.barrier()
        times = []
        for _ in range(steps):
            tic = time.perf_counter()
            fn()
            times.append(time.perf_counter() - tic)
        mine = sum(times) / len(times)
        t = torch.tensor([mine], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return mine, float(t.item())

    host = None
    e2e_bins = bins
    while host is None and e2e_bins >= 1024:
        try:
            host = torch.empty((e2e_bins, x.shape[1]), dtype=torch.int8, pin_memory=True)
        except RuntimeError:
            e2e_bins //= 2
    host.copy_(x[:e2e_bins])
    packed_dev, bits = engine.pack_bits(x[:e2e_bins], cols, k)
    packed = torch.empty(packed_dev.shape, dtype=torch.uint8, pin_memory=True)
    packed.copy_(packed_dev)
    del packed_dev
    torch.cuda.synchronize()
    ntab = k if saliency == 1 else k * k
    d2h = e2e_bins * k * 4 + ntab * 12
    mine_p, t_p = timed(lambda: engine.single_host_packed(packed, cols, k, saliency, bits))
    mine_i, t_i = timed(lambda: engine.single_host(host, cols, k, saliency))
    h2d_p, h2d_i = e2e_bins * int(packed.shape[1]), e2e_bins * int(x.shape[1])
    out = {"value": e2e_bins * world / t_p, "unit": "bins/s", "h2d_bytes_per_step": h2d_p, "d2h_bytes_per_step": d2h,
           "bins_per_gpu": e2e_bins, "steps": steps, "rank0_pcie_GBps": (h2d_p + d2h) / mine_p / 1e9,
           "api": "epi_single_host_packed (C ABI: pinned host matrix in the %d-bit packed transport layout in, tables + "
                  "float32 scores out)" % bits,
           "int8_layout": {"value": e2e_bins * world / t_i, "unit": "bins/s", "h2d_bytes_per_step": h2d_i,
                           "d2h_bytes_per_step": d2h, "rank0_pcie_GBps": (h2d_i + d2h) / mine_i / 1e9,
                           "api": "epi_single_host (int8 host matrix)"}}
    del host, packed
    return out


def run_ours_s3(args, engine, synth, dist, world, rank, local, bins, cols, k, desc):
    """S3 (BASELINE configs[2]): one-hot expansion + tcgen05 int8 Gram (chunked) + finalise + pair terms + scores.
    Parity-test configuration; reported with the tensor-pipe roofline of the Gram kernel."""
    import torch
    if args.bins:
        bins = args.bins
    x = synth.synth_states_device(bins, cols, k, seed=4321 + rank, kind=args.kind)
    plan = engine.s3_plan(bins, cols, k)
    tiles = torch.empty(plan["tile_bytes"] // 4, dtype=torch.int32, device="cuda")
    scores = torch.empty((bins, k), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream()
    gram_ev = []
    keep = {}

    def step(timed):
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        engine.s3_expected_tiles(x, cols, k, tiles=tiles)
        if timed:
            e1.record(stream)
            gram_ev.append((e0, e1))
        if world > 1:
            dist.all_reduce(tiles)
        _, exp3 = engine.s3_finalize(tiles, cols, k, plan["mp"], bins * world, want_counts=False, want_exp=True)
        terms = engine.s3_terms(exp3.reshape(-1), cols, k)
        engine.scores_s3(x, cols, k, terms, out32=scores)
        keep["exp3"] = exp3

    steps = args.steps
    sampler = ClockSampler(local) if rank == 0 else None
    step(False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if sampler:
        sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(steps):
        step(True)
    t1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([t0.elapsed_time(t1) / steps, sum(a.elapsed_time(b) for a, b in gram_ev) / len(gram_ev)],
                      device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step, gram_ms = float(ms[0]), float(ms[1])
    if args.dump_outputs and rank == 0:
        rows = sample_rows(bins)
        dump_outputs(args.dump_outputs, rows, {"scores": take_rows(scores, rows)}, {"expected": keep["exp3"]})
    e2e = None
    if not args.no_e2e:
        # end to end through epi_s3_host: pinned host matrix in, float32 scores out (the 0.9 GB table stays on the device)
        host = torch.empty(x.shape, dtype=torch.int8, pin_memory=True)
        host.copy_(x)
        out = torch.empty((bins, k), dtype=torch.float32, pin_memory=True)
        torch.cuda.synchronize()
        engine.s3_host(host, cols, k, want_exp=False, scores_out=out)
        if world > 1:
            dist.barrier()
        times = []
        for _ in range(2):
            tic = time.perf_counter()
            engine.s3_host(host, cols, k, want_exp=False, scores_out=out)
            times.append(time.perf_counter() - tic)
        t = torch.tensor([sum(times) / len(times)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": bins * world / float(t.item()), "unit": "bins/s", "h2d_bytes_per_step": bins * int(x.shape[1]),
               "d2h_bytes_per_step": bins * k * 4, "steps": 2,
               "api": "epi_s3_host (C ABI: pinned int8 host matrix in, float32 scores out; each rank its own matrix)"}
        del host, out
    if rank == 0:
        ck = cols * k
        useful = bins * ck * (ck + 1)
        peak_tops = 4500.0
        pf = ROOT / "profiles" / "int8_tensor_peak.json"
        src = "datasheet dense int8 4.5 POP/s (B200)"
        if pf.exists():
            try:
                peak_tops = float(json.loads(pf.read_text())["probe_issued_TOPS"])
                src = "measured: same kernel with operand loads disabled (profiles/int8_tensor_peak.json)"
            except Exception:
                pass
        line = {
            "metric": "bins/sec for expected+scores (S3)", "value": bins * world / (ms_per_step * 1e-3), "unit": "bins/s",
            "n_gpus": world, "steps": steps, "warmup": 1, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8 x u8 -> s32 (tensor), f64 scores", "data": "synthetic",
            "config": {"workload": desc, "bins_per_gpu": bins, "biosamples": cols, "states": k, "saliency": 3,
                       "distribution": args.kind, "l2": "one-hot operand panels streamed per 131072-bin chunk"},
            "roofline": {"bound": "tensor", "kernel": "s3_onehot_kernel + s3_gram_kernel (chunked)",
                         "achieved": useful / (gram_ms * 1e-3) / 1e12, "peak": peak_tops, "unit": "TOP/s",
                         "frac": useful / (gram_ms * 1e-3) / 1e12 / peak_tops, "traffic": None, "peak_source": src,
                         "algorithmic_ops_per_launch": useful, "ms_per_launch": gram_ms},
            "e2e": e2e, "gpu_launches": steps * (2 * ((bins + engine.S3_CHUNK_BINS - 1) // engine.S3_CHUNK_BINS) + 4),
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_arm(args, 1, 0, budget_s=20.0)[0]
            except Exception as exc:
                line["cpu_baseline"] = {"error": str(exc)[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_ours_paired(args, engine, synth, dist, world, rank, local, bins, cols, k, desc):
    """Paired mode (BASELINE configs[3]): counts of both groups, expected table of the union (all-reduced), scores A / B,
    delta, quiescence mask, real distances, then P null shuffles per bin (multivariate hypergeometric draws from the group
    counts, scores of the shuffled groups, signed squared null distance).  The reference draws ONE shuffle per bin;
    P = 1000 is the north-star configuration.  Parity-test configuration; reported without a roofline fraction (the null
    stage is bound by the random draws, not by a memory or tensor pipe)."""
    import torch
    if args.bins:
        bins = args.bins
    c1, c2, nperm, batch = 400, 433, 1000, 20
    xa = synth.synth_states_device(bins, c1, k, seed=5 + 10 * rank)
    xb = synth.synth_states_device(bins, c2, k, seed=6 + 10 * rank)
    stream = torch.cuda.current_stream()
    rows = sample_rows(bins, DUMP_ROWS // 64) if args.dump_outputs else None     # 1000 null distances per bin
    last = {}

    def step(nulls=None):
        ca = engine.bin_counts(xa, c1, k)
        cb = engine.bin_counts(xb, c2, k)
        comb = (ca + cb).contiguous()
        n1, _ = engine.expected_tables(comb, c1 + c2, want_s2=False)
        if world > 1:
            dist.all_reduce(n1)
        e = engine.normalize(n1)
        sa, sb = engine.scores_s1(ca, c1, e), engine.scores_s1(cb, c2, e)
        delta, _ = engine.pairwise_combine(sa, sb, None, None)
        mask = engine.quiescent_mask(ca, c1, cb, c2, k - 1)
        dist_real, max_diff = engine.pairwise_real_reduce(delta)
        last.update(expected=e, delta=delta, quiescent=mask, distance=dist_real, max_diff_state=max_diff)
        done = 0
        while done < nperm:
            n = min(batch, nperm - done)
            oa, ob = engine.shuffled_counts_philox(ca, cb, c1, c2, 100 + done, n)
            na = engine.scores_s1(oa.reshape(-1, k), c1, e)
            nb = engine.scores_s1(ob.reshape(-1, k), c2, e)
            _, null = engine.pairwise_combine(None, None, na, nb)
            if nulls is not None:
                nulls.append(take_rows(null.view(n, bins).t(), rows))
            done += n

    steps = args.steps
    sampler = ClockSampler(local) if rank == 0 else None
    step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if sampler:
        sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(steps):
        step()
    t1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([t0.elapsed_time(t1) / steps], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if args.dump_outputs:
        # The null distances of a step are dropped batch by batch, so the last timed step's are taken from one more pass,
        # untimed: the step is deterministic (seeded inputs, null draws keyed by seed and bin).  That pass must reproduce
        # the last timed step's other outputs bit for bit, or the dump would mix two different computations.
        timed = dict(last)
        nulls = []
        step(nulls)
        for name, t in timed.items():
            if not torch.equal(t, last[name]):
                raise RuntimeError("--dump-outputs: the paired step is not deterministic (%s differs between passes)" % name)
        if rank == 0:
            per_bin = {name: take_rows(timed[name], rows) for name in ("delta", "quiescent", "distance", "max_diff_state")}
            per_bin["null_distances"] = torch.cat(nulls, dim=1)
            dump_outputs(args.dump_outputs, rows, per_bin, {"expected": timed["expected"]})
    e2e = None
    if not args.no_e2e:
        # end to end through epi_paired_host with pinned host matrices: tables, delta, quiescence mask and null distances
        # come back to the host.  Headline: ONE null shuffle per bin (what the reference computes); p1000 = the north-star
        # extension (1000 shuffles per bin, 4 bytes x 1000 per bin of null distances cross PCIe).
        ha = torch.empty(xa.shape, dtype=torch.int8, pin_memory=True)
        hb = torch.empty(xb.shape, dtype=torch.int8, pin_memory=True)
        ha.copy_(xa)
        hb.copy_(xb)
        delta_out = torch.empty((bins, k), dtype=torch.float32, pin_memory=True)
        torch.cuda.synchronize()
        res = {}
        for p in (1, nperm):
            null_out = torch.empty((p, bins), dtype=torch.float32, pin_memory=True)
            call = lambda: engine.paired_host(ha, c1, hb, c2, k, 1, k - 1, seed=7, nperm=p, null_out=null_out,
                                              delta_out=delta_out)
            call()
            if world > 1:
                dist.barrier()
            times = []
            for _ in range(2):
                tic = time.perf_counter()
                call()
                times.append(time.perf_counter() - tic)
            t = torch.tensor([sum(times) / len(times)], device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res[p] = {"value": bins * world / float(t.item()), "unit": "bins/s",
                      "h2d_bytes_per_step": bins * int(xa.shape[1] + xb.shape[1]),
                      "d2h_bytes_per_step": bins * (k * 4 + 1 + 4 * p) + k * 12, "null_permutations": p, "steps": 2}
            del null_out
        e2e = dict(res[1], api="epi_paired_host (C ABI: two pinned int8 host matrices in; table, delta, quiescence mask and "
                               "null distances out), one null shuffle per bin as in the reference", p1000=res[nperm])
        del ha, hb, delta_out
    if rank == 0:
        ms_per_step = float(ms[0])
        line = {
            "metric": "bins/sec for paired expected+scores (S1) with %d null permutations per bin" % nperm,
            "value": bins * world / (ms_per_step * 1e-3), "unit": "bins/s", "n_gpus": world, "steps": steps, "warmup": 1,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64+f64", "data": "synthetic",
            "config": {"workload": desc, "bins_per_gpu": bins, "group_sizes": [c1, c2], "states": k, "saliency": 1,
                       "null_permutations": nperm, "bin_permutation_pairs_per_s": bins * world * nperm / (ms_per_step * 1e-3)},
            "roofline": None, "e2e": e2e, "gpu_launches": steps * (12 + (nperm // batch) * 6), "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_arm(args, 1, 0, budget_s=12.0)[0]
            except Exception as exc:
                line["cpu_baseline"] = {"error": str(exc)[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
