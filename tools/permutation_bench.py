"""Per-bin permutation counts (--null-permutations P) on the GPU.  One JSON line per case, with the card's name and power
limit read in the same run.

  kernel  bins x (400 + 433) x 18 group counts resident on the device (rows drawn from 64 count profiles, half of them
          quiescent-like), P shuffles per bin.  S1: the fused kernel (epi_permutation_exceedances_s1) against the composed
          path (epi_shuffled_counts_philox_range + epi_scores_s1 + epi_null_exceedances over bin chunks x permutation
          blocks); S2: the composed path with the tensor-core scores.  The counts of both S1 routes are compared before
          the times are reported.  Wall clock around one call ending in a device synchronise, after a warm-up on 1 % of
          the bins.  pairs_per_s = bins * P / time.
  files   the paired S1 command line file to file on bins x (400 + 433) x 18, with and without --null-permutations P (each
          a fresh process, as a user would run it), wall clock; every other output is compared byte for byte.

    python tools/permutation_bench.py [--out FILE.jsonl] [--bins N] [--perms P] [--skip-files]   (lines go to stdout, and
                                                                                                     to FILE)
"""
import argparse
import gzip
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from epilogos_b200 import engine  # noqa: E402
from epilogos_b200.backend import CudaBackend  # noqa: E402
from epilogos_b200.preprocess import write_matrix  # noqa: E402

C1, C2, K = 400, 433, 18


def card():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return smi[torch.cuda.current_device()] if smi else torch.cuda.get_device_name()


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def profiles(rng):
    """64 (count A, count B) rows: half with one dominant state (quiescent-like), half spread over a few states."""
    rows = []
    for i in range(64):
        p = rng.dirichlet(np.ones(K) * (0.05 if i < 32 else 0.5))
        q = p if i % 3 else rng.dirichlet(np.ones(K) * 0.5)
        rows.append((rng.multinomial(C1, p), rng.multinomial(C2, q)))
    return (torch.tensor(np.array([r[0] for r in rows]).astype(np.int16)),
            torch.tensor(np.array([r[1] for r in rows]).astype(np.int16)))


def composed_s1(ca, cb, dist, exp, P, seed, workspace_bytes=1 << 30):
    """The composed route for S1 (what the backend runs for S2 and for tables wider than the S1 value table)."""
    rows = ca.shape[0]
    k = torch.zeros(rows, dtype=torch.int32, device="cuda")
    pairs = max(1, workspace_bytes // (12 * K))
    chunk = max(1, min(rows, pairs))
    block = max(1, min(P, pairs // chunk))
    for lo in range(0, rows, chunk):
        hi = min(rows, lo + chunk)
        for p0 in range(0, P, block):
            n = min(block, P - p0)
            oa, ob = engine.shuffled_counts_philox_range(ca[lo:hi], cb[lo:hi], C1, C2, seed, p0, n, C1 + C2, bin_offset=lo)
            sa = engine.scores_s1(oa.reshape(-1, K), C1, exp).reshape(n, hi - lo, K)
            sb = engine.scores_s1(ob.reshape(-1, K), C2, exp).reshape(n, hi - lo, K)
            engine.null_exceedances(sa, sb, dist[lo:hi], k[lo:hi])
    return k


def kernel_cases(bins, P, info):
    rng = np.random.default_rng(2026)
    pa, pb = profiles(rng)
    idx = torch.randint(0, 64, (bins,), device="cuda")
    ca, cb = pa.cuda()[idx].contiguous(), pb.cuda()[idx].contiguous()
    be = CudaBackend()
    seed = 0x5EED
    lines = []
    for saliency in (1, 2):
        n1, n2 = engine.expected_tables((ca + cb).contiguous(), C1 + C2, want_s1=saliency == 1, want_s2=saliency == 2)
        exp = engine.normalize(n1 if saliency == 1 else n2)
        sa = be.scores(ca, C1, saliency, exp, perms=C1 * (C1 - 1))
        sb = be.scores(cb, C2, saliency, exp, perms=C2 * (C2 - 1))
        delta, _ = engine.pairwise_combine(sa, sb, None, None)
        dist, _ = engine.pairwise_real_reduce(delta, True)
        del sa, sb, delta

        def backend(lo, hi):
            return be.permutation_exceedances(ca[lo:hi], cb[lo:hi], dist[lo:hi], P, seed, C1, C2, C1 + C2, lo, saliency,
                                              exp, (C1, C2), (C1 * (C1 - 1), C2 * (C2 - 1)))

        warm = max(1, bins // 100)
        backend(0, warm)
        k, t = wall(lambda: backend(0, bins))
        line = dict(case="kernel", saliency=saliency, shape="%d x (%d + %d) x %d" % (bins, C1, C2, K), permutations=P,
                    route="fused" if saliency == 1 else "composed", seconds=round(t, 3),
                    pairs_per_s=float("%.4g" % (bins * P / t)), card=info)
        if saliency == 1:
            composed_s1(ca[:warm], cb[:warm], dist[:warm], exp, P, seed)
            kc, tc = wall(lambda: composed_s1(ca, cb, dist, exp, P, seed))
            line.update(composed_seconds=round(tc, 3), composed_pairs_per_s=float("%.4g" % (bins * P / tc)),
                        speedup=round(tc / t, 2), counts_equal=bool(torch.equal(k, kc)))
            del kc
        line["mean_p"] = round(float(((k.double() + 1) / (P + 1)).mean()), 4)
        lines.append(line)
        print(json.dumps(line), flush=True)
        del k
        torch.cuda.empty_cache()
    return lines


def read_outputs(d, skip):
    return {p.name: (gzip.open(p).read() if p.suffix == ".gz" else p.read_bytes())
            for p in sorted(Path(d).iterdir()) if p.is_file() and skip not in p.name}


def files_case(bins, P, info):
    rng = np.random.default_rng(7)
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        x = rng.integers(0, K, size=(bins, C1 + C2), dtype=np.int8)
        x[rng.random(bins) < 0.5] = K - 1
        x[: bins // 10, :C1] = rng.integers(0, 3, size=(bins // 10, C1))
        for d, cols in (("a", slice(0, C1)), ("b", slice(C1, C1 + C2))):
            (tmp / d).mkdir()
            write_matrix(tmp / d / "epilogos_matrix_chr1.txt.gz", "chr1", np.ascontiguousarray(x[:, cols]), gzip_level=1)
        meta = tmp / "meta.tsv"
        meta.write_text("zero_index\tone_index\tshort_name\tlong_name\n" +
                        "".join("%d\t%d\tS%d\ts%d\n" % (i, i + 1, i + 1, i + 1) for i in range(K)))
        cmd = [sys.executable, "-m", "epilogos_b200.run", "-m", "paired", "-a", str(tmp / "a"), "-b", str(tmp / "b"),
               "-j", str(meta), "-s", "1", "-n"]
        env = dict(os.environ, PYTHONPATH=str(ROOT), EPILOGOS_B200_SEED="1")
        times = {}
        for name, extra in (("plain", []), ("perm", ["--null-permutations", str(P)])):
            t0 = time.perf_counter()
            subprocess.run(cmd + ["-o", str(tmp / name)] + extra, check=True, env=env, stdout=subprocess.DEVNULL, cwd=tmp)
            times[name] = time.perf_counter() - t0
        same = read_outputs(tmp / "plain", "Permutation") == read_outputs(tmp / "perm", "Permutation")
        rows = len(gzip.open(tmp / "perm" / "pairwisePermutation_a_b_s1.txt.gz").read().splitlines())
        return dict(case="files", shape="%d x (%d + %d) x %d" % (bins, C1, C2, K), saliency=1, permutations=P,
                    without_flag_s=round(times["plain"], 2), with_flag_s=round(times["perm"], 2),
                    permutation_rows=rows, other_outputs_identical=bool(same), card=info)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--bins", type=int, default=15_500_000)
    ap.add_argument("--perms", type=int, default=1000)
    ap.add_argument("--file-bins", type=int, default=400_000)
    ap.add_argument("--skip-files", action="store_true")
    a = ap.parse_args()
    info = card()
    lines = kernel_cases(a.bins, a.perms, info)
    if not a.skip_files:
        lines.append(files_case(a.file_bins, a.perms, info))
        print(json.dumps(lines[-1]), flush=True)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
