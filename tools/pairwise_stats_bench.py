"""Timing of the paired statistics stage (csrc/pairwise_stats.cu) at genome scale on one GPU, with the card's name and
power limit read in the same run.  One JSON line:

  fit_ms            null subsampling + gennorm fits, T trials x S points, from a pool of `bins` null distances
  pvalues_ms        p-values of `bins` distances;  bh_ms  Benjamini-Hochberg over them
  metrics_write_s   pairwiseMetrics text of `bins` rows (8 columns) through the native gzip writer (host wall clock)
  scipy_fit_s       one scipy.stats.gennorm.fit of trial 0's S points on the host (the CPU arm), mean of `--scipy-fits`
Inputs are seeded: the pool and the distances are gennorm(beta = 0.4) draws with 14 % exact zeros, like real null
distances.  Device times are CUDA events around `--reps` repetitions after one warm-up; the 62 MB pool stays in L2.

    python tools/pairwise_stats_bench.py [--bins 15500000] [--trials 101] [--size 100000] [--out FILE]
"""
import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import scipy.stats
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from epilogos_b200 import engine, writer  # noqa: E402
from oracle import pairwise_stats_oracle as pso  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--bins", type=int, default=15_500_000)
ap.add_argument("--trials", type=int, default=101)
ap.add_argument("--size", type=int, default=100_000)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--scipy-fits", type=int, default=3)
ap.add_argument("--out", type=str, default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("pairwise_stats_bench needs a CUDA device")


def timed_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1) / reps


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
rng = np.random.default_rng(2026)
vals = (scipy.stats.gennorm.rvs(0.4, size=a.bins, random_state=rng) * 0.05).astype(np.float32)
vals[rng.random(a.bins) < 0.14] = 0.0
pool = torch.from_numpy(vals).cuda()
dist = torch.from_numpy(np.roll(vals, 12345)).cuda()


def fit():
    _, samples = engine.null_subsample(pool, a.trials, a.size, 7)
    return engine.gennorm_fit(samples)


(params, status), fit_ms = timed_ms(fit, a.reps)
params = params.cpu().numpy()
chosen = pso.median_trial(params[:, 3])
beta, loc, scale = params[chosen, :3]
p, pv_ms = timed_ms(lambda: engine.gennorm_pvalues(dist, beta, loc, scale), a.reps)
q, bh_ms = timed_ms(lambda: engine.bh_adjust(p), a.reps)

idx, _ = engine.null_subsample(pool, 1, a.size, 7)
points = vals[idx.cpu().numpy()[0]]
t0 = time.perf_counter()
for _ in range(a.scipy_fits):
    ref = pso.fit(points)
scipy_s = (time.perf_counter() - t0) / a.scipy_fits

n = a.bins
loc_cols = dict(chrom=np.array(["chr1"] * n, dtype=object), start=np.arange(n, dtype=np.int64) * 200,
                end=np.arange(n, dtype=np.int64) * 200 + 200)
md = rng.integers(1, 19, n).astype(np.int32)
with tempfile.TemporaryDirectory() as tmp:
    t0 = time.perf_counter()
    writer.write_metrics_text(Path(tmp) / "m.txt.gz", loc_cols, ["S%d" % i for i in range(1, 19)], md,
                              dist.cpu().numpy(), p.cpu().numpy(), q.cpu().numpy())
    write_s = time.perf_counter() - t0

line = dict(tool="pairwise_stats_bench", device=smi, bins=n, trials=a.trials, size=a.size, reps=a.reps,
            fit_ms=round(fit_ms, 3), pvalues_ms=round(pv_ms, 3), bh_ms=round(bh_ms, 3),
            metrics_write_s=round(write_s, 3), scipy_fit_s=round(scipy_s, 4),
            scipy_fits_for_all_trials_s=round(scipy_s * a.trials, 2),
            fit_iterations_max=int(status[:, 0].max().item()), fit_converged=int(status[:, 1].sum().item()),
            chosen=dict(trial=chosen, beta=float(beta), loc=float(loc), scale=float(scale)),
            trial0_device_minus_scipy=[float(params[0, i] - ref[i]) for i in range(3)])
print(json.dumps(line), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, "a") as f:
        f.write(json.dumps(line) + "\n")
