"""The region null (--roi-permutations P) on the GPU.  One JSON line per case, with the card's name and power limit read in
the same run.

For bins x (400 + 433) x 18 labels from epilogos_b200.synth ("realistic" and "uniform"), resident on the device, and P
splits: wall clock of CudaBackend.region_maxima_paired (G = 2) or region_maxima_multigroup (G = 3: 278 + 278 + 277), S1
or S2, around one call ending in a device synchronise, after a warm-up on 50 000 bins.  Per-kernel times come from CUDA
events around each engine call of that same call, summed by kind (epi_split_counts validates its bitsets on the host
after a stream synchronise, so its time includes that wait): split counts (epi_split_counts), scores (the S1 / S2 score
kernels of every group), statistic (epi_pairwise_combine + epi_pairwise_real_reduce + abs, or epi_multigroup_stat),
window maxima (epi_window_max); "other" is the rest of the wall clock (host draws of the splits, bitset uploads,
allocation).

    python tools/region_permutation_bench.py [--out FILE.jsonl] [--bins N ...] [--perms P] [--kinds realistic uniform]
"""
import argparse
import json
import subprocess
import sys
import time
from collections import defaultdict
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from epilogos_b200 import engine  # noqa: E402
from epilogos_b200.backend import CudaBackend  # noqa: E402
from epilogos_b200.synth import synth_states_device  # noqa: E402

K, W = 18, 125
SIZES = {2: (400, 433), 3: (278, 278, 277)}


def card():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return smi[torch.cuda.current_device()] if smi else torch.cuda.get_device_name()


class KernelTimes:
    """CUDA events around the engine entry points of one call, summed per kind."""
    KINDS = {"split_counts": "split counts", "scores_s1": "scores", "scores_s2": "scores",
             "pairwise_combine": "statistic", "pairwise_real_reduce": "statistic", "multigroup_stat": "statistic",
             "window_max": "window maxima"}

    def __init__(self):
        self.events = defaultdict(list)
        self.saved = {}

    def __enter__(self):
        for name, kind in self.KINDS.items():
            fn = getattr(engine, name)
            self.saved[name] = fn

            def timed(*a, _fn=fn, _kind=kind, **k):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                out = _fn(*a, **k)
                e.record()
                self.events[_kind].append((s, e))
                return out
            setattr(engine, name, timed)
        return self

    def __exit__(self, *exc):
        for name, fn in self.saved.items():
            setattr(engine, name, fn)

    def totals(self):
        torch.cuda.synchronize()
        return {k: sum(s.elapsed_time(e) for s, e in v) / 1e3 for k, v in self.events.items()}


def run(be, x, G, saliency, exp, P):
    sizes = SIZES[G]
    fn = be.region_maxima_paired if G == 2 else be.region_maxima_multigroup
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with KernelTimes() as kt:
        m = fn(x, None, sizes, K, W, P, 1234, saliency, exp)
        torch.cuda.synchronize()
    return m, time.perf_counter() - t0, kt.totals()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--bins", type=int, nargs="+", default=[1_250_000, 15_500_000])
    ap.add_argument("--perms", type=int, default=1000)
    ap.add_argument("--kinds", nargs="+", default=["realistic", "uniform"])
    args = ap.parse_args()
    be = CudaBackend()
    who = card()
    N = sum(SIZES[2])
    for bins in args.bins:
        for kind in args.kinds:
            x = synth_states_device(bins, N, K, seed=7, kind=kind)
            union = engine.bin_counts(x, N, K)
            n1, n2 = engine.expected_tables(union, N)
            exps = {1: engine.normalize(n1), 2: engine.normalize(n2)}
            del union
            for saliency in (1, 2):
                for G in (2, 3):
                    run(be, x[:50_000].contiguous(), G, saliency, exps[saliency], 8)     # warm-up of every shape
                    m, secs, kern = run(be, x, G, saliency, exps[saliency], args.perms)
                    line = dict(case="region_null", card=who, bins=bins, cols=N, states=K, kind=kind, saliency=saliency,
                                groups=G, window=W, perms=args.perms, wall_s=round(secs, 3),
                                kernel_s={k: round(v, 3) for k, v in sorted(kern.items())},
                                other_s=round(secs - sum(kern.values()), 3),
                                max_of_maxima=int(m.max().item()))
                    print(json.dumps(line), flush=True)
                    if args.out:
                        with open(args.out, "a") as f:
                            f.write(json.dumps(line) + "\n")
            del x
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
