"""Multi-group permutation counts on the GPU.  One JSON line per case, with the card's name and power limit read in the
same run.

  bins x 833 x 18 group counts resident on the device (rows drawn from 64 count profiles, half of them quiescent-like),
  the 833 biosamples split into G groups.  Cases:
    s1_fused       epi_multigroup_exceedances_s1, G = 2, 4, 8, P shuffles per bin
    s1_composed    sampler + epi_scores_s1 per group + epi_multigroup_null_exceedances (CudaBackend's composed loop, 1 GiB
                   cap) for G = 4 at --composed-perms shuffles; its counts are compared with the fused kernel's first
                   --composed-perms shuffles, and seconds_at_P scales its time linearly to P
    s2_composed    the same loop with the tensor-core S2 scores, G = 4, --composed-perms shuffles, scaled to P
    stat           epi_multigroup_stat alone on the G = 4 score arrays
    paired_fused   epi_permutation_exceedances_s1 of the paired mode on the G = 2 split, P shuffles: the baseline
  Wall clock around one call ending in a device synchronise, after a warm-up on 1 % of the bins.
    files          the command line file to file on --files-bins x 833 x 18, S1, P = 100: one --multigroup of 4 groups
                   against one run with the 6 --compare pairs it replaces (each a fresh process, as a user would run it)

    python tools/multigroup_bench.py [--out FILE.jsonl] [--bins N] [--perms P] [--composed-perms Q] [--files-bins N]
"""
import argparse
import json
import os
import subprocess
import tempfile
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from epilogos_b200 import engine  # noqa: E402
from epilogos_b200.backend import CudaBackend  # noqa: E402

WIDTH, K = 833, 18


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


def split(width, parts):
    base, extra = divmod(width, parts)
    return [base + (1 if g >= parts - extra else 0) for g in range(parts)]


def group_counts(rng, bins, sizes):
    """[G, bins, K] counts: each bin is one of 64 label profiles, each group a multinomial draw from it (a third of the
    profiles give one group its own distribution)."""
    G = len(sizes)
    prof = []
    for i in range(64):
        p = rng.dirichlet(np.ones(K) * (0.05 if i < 32 else 0.5))
        q = p if i % 3 else rng.dirichlet(np.ones(K) * 0.5)
        prof.append([rng.multinomial(n, q if g == G - 1 else p) for g, n in enumerate(sizes)])
    prof = torch.tensor(np.array(prof).astype(np.int16)).cuda()          # [64, G, K]
    idx = torch.randint(0, 64, (bins,), device="cuda")
    return prof[idx].permute(1, 0, 2).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--bins", type=int, default=15_500_000)
    ap.add_argument("--perms", type=int, default=1000)
    ap.add_argument("--composed-perms", type=int, default=8)
    ap.add_argument("--files-bins", type=int, default=400_000)
    a = ap.parse_args()
    be = CudaBackend()
    dev = card()
    lines = []
    rng = np.random.default_rng(0)
    seed, P, Q, bins = 0x5EED, a.perms, a.composed_perms, a.bins

    def emit(**kw):
        kw.update(card=dev, bins=bins, width=WIDTH, states=K)
        line = json.dumps(kw)
        print(line, flush=True)
        lines.append(line)

    for G in (2, 4, 8):
        sizes = split(WIDTH, G)
        cnt = group_counts(rng, bins, sizes)
        union = cnt.sum(dim=0, dtype=torch.int32).to(torch.int16).contiguous()
        n1, n2 = engine.expected_tables(union, WIDTH)
        del union
        e1, e2 = engine.normalize(n1), engine.normalize(n2)
        warm = max(1, bins // 100)
        be.multigroup_stat(cnt[:, :warm], sizes, 1, e1)
        t, _, _, _ = be.multigroup_stat(cnt, sizes, 1, e1)
        if G == 4:
            sc = torch.stack([engine.scores_s1(cnt[g].contiguous(), n, e1) for g, n in enumerate(sizes)])
            engine.multigroup_stat(sc, sizes)
            _, sec = wall(lambda: engine.multigroup_stat(sc, sizes))
            emit(case="stat", groups=G, seconds=sec, bytes_read=sc.numel() * 4)
            del sc

        def fused(n, lo=0, hi=bins):
            k = torch.zeros(hi - lo, dtype=torch.int32, device="cuda")
            return engine.multigroup_exceedances_s1(cnt[:, lo:hi], sizes, seed, 0, n, lo, e1, t[lo:hi].contiguous(), k)

        fused(P, 0, warm)
        k, sec = wall(lambda: fused(P))
        emit(case="s1_fused", groups=G, perms=P, seconds=sec, pairs_per_s=bins * P / sec, mean_k=float(k.double().mean()))
        if G == 2:
            dist = (torch.rand(bins, device="cuda") * 0.01).contiguous()

            def paired(n, lo=0, hi=bins):
                k = torch.zeros(hi - lo, dtype=torch.int32, device="cuda")
                return engine.permutation_exceedances_s1(cnt[0, lo:hi].contiguous(), cnt[1, lo:hi].contiguous(), sizes[0],
                                                         sizes[1], seed, 0, n, WIDTH, lo, e1, sizes[0], sizes[1],
                                                         dist[lo:hi].contiguous(), k)
            paired(P, 0, warm)
            _, sec = wall(lambda: paired(P))
            emit(case="paired_fused", groups=2, perms=P, seconds=sec, pairs_per_s=bins * P / sec)
        if G == 4:
            kq = fused(Q)
            composed = lambda: engine_composed(be, cnt, sizes, t, Q, seed, 1, e1)   # noqa: E731
            engine_composed(be, cnt[:, :warm], sizes, t[:warm].contiguous(), Q, seed, 1, e1)
            kc, sec = wall(composed)
            emit(case="s1_composed", groups=G, perms=Q, seconds=sec, seconds_at_P=sec * P / Q, perms_scaled_to=P,
                 equal_to_fused=bool(torch.equal(kc, kq)))
            t2, _, _, _ = be.multigroup_stat(cnt, sizes, 2, e2)
            engine_composed(be, cnt[:, :warm], sizes, t2[:warm].contiguous(), Q, seed, 2, e2)
            _, sec = wall(lambda: engine_composed(be, cnt, sizes, t2, Q, seed, 2, e2))
            emit(case="s2_composed", groups=G, perms=Q, seconds=sec, seconds_at_P=sec * P / Q, perms_scaled_to=P)
        del cnt, t
        torch.cuda.empty_cache()
    if a.files_bins:
        emit(**files_case(a.files_bins))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("\n".join(lines) + "\n")


def files_case(bins, P=100):
    from epilogos_b200.preprocess import write_matrix
    rng = np.random.default_rng(7)
    sizes = split(WIDTH, 4)
    edges = np.concatenate([[0], np.cumsum(sizes)])
    names = ["t%d" % g for g in range(4)]
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        x = rng.integers(0, K, size=(bins, WIDTH), dtype=np.int8)
        x[rng.random(bins) < 0.5] = K - 1
        x[: bins // 10, : sizes[0]] = rng.integers(0, 3, size=(bins // 10, sizes[0]))
        (tmp / "in").mkdir()
        write_matrix(tmp / "in" / "epilogos_matrix_chr1.txt.gz", "chr1", x, gzip_level=1)
        (tmp / "g.tsv").write_text("".join("%s\t%d-%d\n" % (n, edges[g] + 1, edges[g + 1]) for g, n in enumerate(names)))
        meta = tmp / "meta.tsv"
        meta.write_text("zero_index\tone_index\tshort_name\tlong_name\n" +
                        "".join("%d\t%d\tS%d\ts%d\n" % (i, i + 1, i + 1, i + 1) for i in range(K)))
        cmd = [sys.executable, "-m", "epilogos_b200.run", "-m", "paired", "-i", str(tmp / "in"), "-j", str(meta), "-s", "1",
               "--groups", str(tmp / "g.tsv"), "--null-permutations", str(P)]
        env = dict(os.environ, PYTHONPATH=str(ROOT), EPILOGOS_B200_SEED="1")
        pairs = ["%s:%s" % (names[i], names[j]) for i in range(4) for j in range(i + 1, 4)]
        times = {}
        for name, extra in (("multigroup", ["--multigroup", ",".join(names)]),
                            ("compare6", [v for pr in pairs for v in ("--compare", pr)])):
            t0 = time.perf_counter()
            subprocess.run(cmd + ["-o", str(tmp / name)] + extra, check=True, env=env, stdout=subprocess.DEVNULL, cwd=tmp)
            times[name] = time.perf_counter() - t0
        wrote = (tmp / "multigroup" / "_".join(names) / ("multigroupMetrics_%s_s1.txt.gz" % "_".join(names))).exists()
        return dict(case="files", shape="%d x %d x %d" % (bins, WIDTH, K), groups=4, saliency=1, perms=P,
                    multigroup_s=round(times["multigroup"], 2), compare6_s=round(times["compare6"], 2), metrics_written=wrote)


def engine_composed(be, cnt, sizes, t, nperm, seed, saliency, exp):
    """CudaBackend's composed loop, whatever the route it would pick for S1."""
    fits = engine.multigroup_s1_fused_fits
    engine.multigroup_s1_fused_fits = lambda *_: False
    try:
        return be.multigroup_exceedances(cnt, sizes, t, nperm, seed, 0, saliency, exp)
    finally:
        engine.multigroup_s1_fused_fits = fits


if __name__ == "__main__":
    main()
