"""Small shapes through every kernel of the S1 / S2 / S3 / paired path and the packed transport layout, for
compute-sanitizer runs:
    compute-sanitizer --tool memcheck  python tools/sanitize_small.py
    compute-sanitizer --tool racecheck python tools/sanitize_small.py --race      (fewer shapes: racecheck is slow)
"""
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from epilogos_b200 import engine  # noqa: E402

race = "--race" in sys.argv
rng = np.random.default_rng(0)
shapes = ((300, 40, 18), (129, 300, 15), (70, 13, 6), (260, 127, 15), (140, 100, 18))
for bins, cols, k in (shapes[:1] + shapes[3:4] if race else shapes):
    x = rng.integers(0, k, size=(bins, cols)).astype(np.int8)
    xh = engine.pack_states(x)
    xd = xh.cuda()
    cnt = engine.bin_counts(xd, cols, k)                                     # K1 (incl. the one-box small-row variant)
    n1, n2 = engine.expected_tables(cnt, cols)                               # K2 (tcgen05 Gram of the count bytes)
    e1, e2 = engine.normalize(n1), engine.normalize(n2 + 1)                  # K4
    engine.scores_s1(cnt, cols, e1, want64=True)                             # K5-S1 value table + look-up
    engine.scores_s2(cnt, cols, e2, want64=True)                             # K5-S2 tensor cores (kind::i8)
    engine.scores_s2(cnt, cols, engine.normalize(n2), want64=True, mode=1)   # DIRECT
    packed, bits = engine.pack_bits(xd, cols, k)                             # packed transport layout
    back = engine.unpack_bits(packed, cols, bits)
    assert torch.equal(back[:, :cols], xd[:, :cols])
    hp, _ = engine.pack_bits_host(xh, cols, k)
    engine.single_host_packed(hp, cols, k, 2, bits)
    engine.single_host(xh, cols, k, 1)
    if cols <= 40:
        tiles, plan = engine.s3_expected_tiles(xd, cols, k)                  # one-hot + two-CTA tcgen05 Gram
        counts, exp = engine.s3_finalize(tiles, cols, k, plan["mp"], bins)
        terms = engine.s3_terms(exp.reshape(-1), cols, k)
        engine.scores_s3(xd, cols, k, terms, want64=True)
        engine.s3_host(xh, cols, k)
    # paired
    c1 = cols // 2
    xa, xb = engine.pack_states(x[:, :c1]).cuda(), engine.pack_states(x[:, c1:]).cuda()
    ca, cb = engine.bin_counts(xa, c1, k), engine.bin_counts(xb, cols - c1, k)
    perm = torch.from_numpy(np.argsort(rng.random((bins, cols)), axis=1).astype(np.int32)).cuda()
    engine.shuffled_counts_perm(xa, c1, xb, cols - c1, perm, k, c1, cols - c1)
    oa, ob = engine.shuffled_counts_philox(ca, cb, c1, cols - c1, seed=3, nperm=3)
    sa, sb = engine.scores_s1(ca, c1, e1), engine.scores_s1(cb, cols - c1, e1)
    delta, _ = engine.pairwise_combine(sa, sb, None, None)
    engine.pairwise_combine(None, None, engine.scores_s1(oa.reshape(-1, k), c1, e1), engine.scores_s1(ob.reshape(-1, k), cols - c1, e1))
    engine.quiescent_mask(ca, c1, cb, cols - c1, k - 1)
    engine.pairwise_real_reduce(delta)
    engine.paired_host(engine.pack_states(x[:, :c1]), c1, engine.pack_states(x[:, c1:]), cols - c1, k, 1, k - 1, nperm=2)
    # permutation counts: range sampler, counting step, fused S1 kernel (1, 8 and 32 threads per bin)
    dist, _ = engine.pairwise_real_reduce(delta)
    pa, pb = engine.shuffled_counts_philox_range(ca, cb, c1, cols - c1, 3, 5, 3, cols, bin_offset=7)
    kk = torch.zeros(bins, dtype=torch.int32, device="cuda")
    engine.null_exceedances(engine.scores_s1(pa.reshape(-1, k), c1, e1).reshape(3, bins, k),
                            engine.scores_s1(pb.reshape(-1, k), cols - c1, e1).reshape(3, bins, k), dist, kk)
    for n in (3, 9, 40):
        engine.permutation_exceedances_s1(ca, cb, c1, cols - c1, 3, 0, n, cols, 7, e1, c1, cols - c1, dist, kk)
    torch.cuda.synchronize()
    print("ok", bins, cols, k, flush=True)
print("done")
