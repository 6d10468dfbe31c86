"""Stratified permutations (--strata) on the GPU.  One JSON line per case, with the card's name and power limit read in the
same run.

  fused   bins x (400 + 433) x 18 counts resident on the device, P = 1000 shuffles per bin: the unstratified fused S1 kernel
          (epi_permutation_exceedances_s1) against the stratified one (epi_stratified_exceedances_s1) with H = 1, 4, 16
          and 64 strata, each group split evenly over the strata.  Rows come from 64 count profiles drawn per stratum (half
          with one dominant state).  Repeats alternate the two kernels; every time is a wall clock around one call ending
          in a device synchronise, after a warm-up on 1 % of the bins.  At H = 1 the counts of both kernels are compared.
  count   the per-stratum count pass (epi_group_counts over a bins x 833 label matrix, one column list per stratum).
  s2      the composed S2 path with strata (CudaBackend.permutation_exceedances: stratified sampler + tensor-core scores +
          epi_null_exceedances), H = 4, P = 100, against the same path without strata.

    python tools/strata_bench.py [--out FILE.jsonl] [--bins N] [--perms P] [--repeats R]
"""
import argparse
import json
import subprocess
import sys
import time
import types
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from epilogos_b200 import engine  # noqa: E402
from epilogos_b200.backend import CudaBackend  # noqa: E402

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


def split(n, H):
    return [n // H + (1 if h < n % H else 0) for h in range(H)]


def strata_inputs(H, bins, seed):
    """(sizes [H][2], cnt_h [H, bins, K], cnt_a, cnt_b) on the device: 64 profiles of per-stratum counts, rows drawn from
    them."""
    rng = np.random.default_rng(seed)
    sizes = [list(v) for v in zip(split(C1, H), split(C2, H))]
    a = np.zeros((H, 64, K), dtype=np.int64)
    b = np.zeros((H, 64, K), dtype=np.int64)
    for i in range(64):
        for h, (na, nb) in enumerate(sizes):
            p = rng.dirichlet(np.ones(K) * (0.05 if i < 32 else 0.5))
            q = p if i % 3 else rng.dirichlet(np.ones(K) * 0.5)
            a[h, i], b[h, i] = rng.multinomial(na, p), rng.multinomial(nb, q)
    idx = torch.from_numpy(rng.integers(0, 64, size=bins)).cuda()
    dev = lambda v: torch.from_numpy(v.astype(np.int16)).cuda()
    cnt_h = dev(a + b)[:, idx].contiguous()
    return sizes, cnt_h, dev(a.sum(axis=0))[idx].contiguous(), dev(b.sum(axis=0))[idx].contiguous()


def real_dist(ca, cb, exp):
    delta, _ = engine.pairwise_combine(engine.scores_s1(ca, C1, exp), engine.scores_s1(cb, C2, exp))
    return engine.pairwise_real_reduce(delta, True)[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--bins", type=int, default=1250000)
    ap.add_argument("--perms", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    engine.device_info()
    name = card()
    lines = []

    def emit(rec):
        rec.update(card=name, tool="tools/strata_bench.py")
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    bins, P = args.bins, args.perms
    shape = "%d x (%d + %d) x %d" % (bins, C1, C2, K)
    for H in (1, 4, 16, 64):
        sizes, cnt_h, ca, cb = strata_inputs(H, bins, seed=H)
        exp = (cnt_h.sum(dim=(0, 1), dtype=torch.int64).double() / (bins * (C1 + C2))).float().contiguous()
        dist = real_dist(ca, cb, exp)
        warm = max(8, bins // 100)

        def plain(n=bins):
            k = torch.zeros(n, dtype=torch.int32, device="cuda")
            return engine.permutation_exceedances_s1(ca[:n], cb[:n], C1, C2, 7, 0, P, C1 + C2, 0, exp, C1, C2, dist[:n], k)

        def strat(n=bins):
            k = torch.zeros(n, dtype=torch.int32, device="cuda")
            return engine.stratified_exceedances_s1(cnt_h[:, :n], sizes, ca[:n], cb[:n], 7, 0, P, 0, exp, C1, C2,
                                                    dist[:n], k)
        plain(warm), strat(warm)
        times = {"plain": [], "strata": []}
        k_plain = k_strat = None
        for r in range(args.repeats):
            for which in (("plain", "strata") if r % 2 == 0 else ("strata", "plain")):
                k, t = wall(plain if which == "plain" else strat)
                times[which].append(t)
                if which == "plain":
                    k_plain = k
                else:
                    k_strat = k
        rec = dict(case="fused", saliency=1, shape=shape, permutations=P, strata=H,
                   plain_seconds=[round(t, 4) for t in times["plain"]],
                   strata_seconds=[round(t, 4) for t in times["strata"]],
                   ratio_median=round(float(np.median(times["strata"]) / np.median(times["plain"])), 4),
                   mean_p_strata=round(float(((1.0 + k_strat.double()) / (P + 1)).mean()), 4))
        if H == 1:
            rec["counts_equal_unstratified"] = bool(torch.equal(k_plain, k_strat))
        emit(rec)
        del cnt_h, ca, cb

    # the per-stratum count pass over a label matrix on the device
    x = torch.randint(0, K, (bins, 848), dtype=torch.int8, device="cuda")
    for H in (1, 4, 16, 64):
        cols = np.array_split(np.random.default_rng(H).permutation(C1 + C2), H)
        engine.group_counts(x[:1024], C1 + C2, K, cols)
        ts = [wall(lambda: engine.group_counts(x, C1 + C2, K, cols))[1] for _ in range(args.repeats)]
        emit(dict(case="count", shape="%d x %d x %d" % (bins, C1 + C2, K), strata=H,
                  seconds=[round(t, 4) for t in ts]))
    del x

    # the composed S2 path, H = 4, P = 100
    be = CudaBackend()
    sizes, cnt_h, ca, cb = strata_inputs(4, bins, seed=44)
    union = (ca + cb)
    n2 = engine.expected_tables(union, C1 + C2, want_s1=False)[1]
    exp2 = engine.normalize(n2)
    sa = engine.scores_s2(ca, C1, exp2)
    sb = engine.scores_s2(cb, C2, exp2)
    delta, _ = engine.pairwise_combine(sa, sb)
    dist = engine.pairwise_real_reduce(delta, True)[0]
    lay = types.SimpleNamespace(counts=cnt_h, sizes=sizes)
    P2 = 100

    def run(strata):
        extra = {} if strata is None else {"strata": strata}
        return be.permutation_exceedances(ca, cb, dist, P2, 7, C1, C2, C1 + C2, 0, 2, exp2, (C1, C2),
                                          (C1 * (C1 - 1), C2 * (C2 - 1)), **extra)
    run(None), run(lay)
    times = {"plain": [], "strata": []}
    for r in range(args.repeats):
        for which in (("plain", "strata") if r % 2 == 0 else ("strata", "plain")):
            times[which].append(wall(lambda: run(None if which == "plain" else lay))[1])
    emit(dict(case="s2", saliency=2, shape=shape, permutations=P2, strata=4,
              plain_seconds=[round(t, 4) for t in times["plain"]],
              strata_seconds=[round(t, 4) for t in times["strata"]],
              ratio_median=round(float(np.median(times["strata"]) / np.median(times["plain"])), 4)))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
