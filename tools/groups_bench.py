"""Column-group counts on the GPU, and a --groups run against separate runs on pre-cut files.  One JSON line per case, with
the card's name and power limit read in the same run.

  kernel  epi_group_counts on a resident random matrix vs the composition it replaces (epi_gather_columns per group, then
          epi_bin_counts) and vs K1 on the whole matrix; CUDA events over `--iters` launches after a warm-up.  The counts of
          both routes are checked equal before timing.  floor_ms = (bins * C bytes read + groups * bins * K * 2 bytes
          written) / 7.7 TB/s, the HBM data-sheet bandwidth of one B200; floor_share = floor_ms / group_counts_ms.
  files   one `--groups` S1 run with 4 disjoint groups of a bins x C TSV.gz against 4 runs on the pre-cut column-subset
          files (each a fresh process, as a user would run them), wall clock; the outputs are compared byte for byte.

    python tools/groups_bench.py [--out FILE.jsonl] [--iters 20] [--skip-files]      (lines go to stdout, and to FILE)
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
from epilogos_b200.preprocess import write_matrix  # noqa: E402

HBM_BPS = 7.7e12


def card():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return smi[torch.cuda.current_device()] if smi else torch.cuda.get_device_name()


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def group_sets(cols, rng):
    def disjoint(n):
        return [np.arange(i * cols // n, (i + 1) * cols // n) for i in range(n)]
    four = disjoint(4)
    scattered = [np.sort(rng.choice(cols, size=cols // 4, replace=False)) for _ in range(3)]
    return {"2_disjoint": disjoint(2), "4_disjoint": disjoint(4), "8_disjoint": disjoint(8),
            "8_overlapping": four + [np.concatenate(four)] + scattered}


def kernel_case(x, cols, k, name, groups, iters, info):
    bins = x.shape[0]
    got = engine.group_counts(x, cols, k, groups)
    subs = [engine.gather_columns(x, cols, g) for g in groups]
    equal = all(torch.equal(got[i], engine.bin_counts(s, len(g), k)) for i, (s, g) in enumerate(zip(subs, groups)))
    del subs
    torch.cuda.empty_cache()
    # the composition keeps one gathered matrix at a time (what it would need per group)
    def composition():
        for g in groups:
            engine.bin_counts(engine.gather_columns(x, cols, g), len(g), k)
    out = torch.empty_like(got)
    t_group = timed(lambda: engine.group_counts(x, cols, k, groups), iters)
    t_comp = timed(composition, max(3, iters // 4))
    t_k1 = timed(lambda: engine.bin_counts(x, cols, k, out=out[0]), iters)
    moved = bins * cols + len(groups) * bins * k * 2
    listed = sum(len(g) for g in groups)
    floor_ms = moved / HBM_BPS * 1e3
    return dict(case="kernel", shape="%d x %d x %d" % (bins, cols, k), groups=name, n_groups=len(groups),
                listed_columns=listed, counts_equal=bool(equal), group_counts_ms=round(t_group, 4),
                gather_plus_k1_ms=round(t_comp, 4), k1_full_matrix_ms=round(t_k1, 4),
                speedup_vs_composition=round(t_comp / t_group, 2), bytes_moved=moved, floor_ms=round(floor_ms, 4),
                floor_share=round(floor_ms / t_group, 3), card=info)


def read_outputs(d):
    out = {}
    for p in sorted(Path(d).rglob("*")):
        if p.is_file():
            out[str(p.relative_to(d))] = gzip.open(p).read() if p.suffix == ".gz" else p.read_bytes()
    return out


def files_case(bins, cols, k, info):
    rng = np.random.default_rng(7)
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        x = rng.integers(0, k, size=(bins, cols), dtype=np.int8)
        x[rng.random(bins) < 0.5] = k - 1
        inp = tmp / "in"
        inp.mkdir()
        write_matrix(inp / "epilogos_matrix_chr1.txt.gz", "chr1", x, gzip_level=1)
        groups = [np.arange(i * cols // 4, (i + 1) * cols // 4) for i in range(4)]
        names = ["g%d" % i for i in range(4)]
        (tmp / "groups.tsv").write_text("".join("%s\t%d-%d\n" % (n, g[0] + 1, g[-1] + 1) for n, g in zip(names, groups)))
        for n, g in zip(names, groups):
            (tmp / "cut" / n).mkdir(parents=True)
            write_matrix(tmp / "cut" / n / "epilogos_matrix_chr1.txt.gz", "chr1", np.ascontiguousarray(x[:, g]), gzip_level=1)
        meta = tmp / "meta.tsv"
        meta.write_text("zero_index\tone_index\tshort_name\tlong_name\n" +
                        "".join("%d\t%d\tS%d\ts%d\n" % (i, i + 1, i + 1, i + 1) for i in range(k)))
        cmd = [sys.executable, "-m", "epilogos_b200.run", "-j", str(meta), "-s", "1"]
        env = dict(os.environ, PYTHONPATH=str(ROOT))
        t0 = time.perf_counter()
        subprocess.run(cmd + ["-i", str(inp), "-o", str(tmp / "grouped"), "--groups", str(tmp / "groups.tsv")], check=True,
                       env=env, stdout=subprocess.DEVNULL, cwd=tmp)
        t_groups = time.perf_counter() - t0
        t0 = time.perf_counter()
        for n in names:
            subprocess.run(cmd + ["-i", str(tmp / "cut" / n), "-o", str(tmp / "separate" / n)], check=True, env=env,
                           stdout=subprocess.DEVNULL, cwd=tmp)
        t_sep = time.perf_counter() - t0
        same = read_outputs(tmp / "grouped") == read_outputs(tmp / "separate")
        return dict(case="files", shape="%d x %d x %d" % (bins, cols, k), saliency=1, n_groups=4,
                    groups_run_s=round(t_groups, 2), separate_runs_s=round(t_sep, 2),
                    speedup=round(t_sep / t_groups, 2), outputs_identical=bool(same), card=info)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--bins", type=int, default=15_500_000)
    ap.add_argument("--file-bins", type=int, default=400_000)
    ap.add_argument("--skip-files", action="store_true")
    a = ap.parse_args()
    info = card()
    lines = []
    rng = np.random.default_rng(2026)
    for cols, k, sets in ((833, 18, None), (127, 15, "2_disjoint")):
        x = torch.randint(0, k, (a.bins, engine.pitch_for(cols)), dtype=torch.int8, device="cuda")
        x[:, cols:] = 0
        for name, groups in group_sets(cols, rng).items():
            if sets is None or name == sets:
                lines.append(kernel_case(x, cols, k, name, groups, a.iters, info))
                print(json.dumps(lines[-1]), flush=True)
        del x
        torch.cuda.empty_cache()
    if not a.skip_files:
        lines.append(files_case(a.file_bins, 833, 18, info))
        print(json.dumps(lines[-1]), flush=True)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
