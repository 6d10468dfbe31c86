"""S3 (-s 3) kernels against independent float64 references on every bin, every tile and every launch variant.

K3 (one-hot expansion + tcgen05 Gram) and epi_s3_finalize are compared with OH^T OH formed by torch in float64 from the
one-hot OH[b][i*K + a] = (x[b, i] == a): sums of 0/1 products below 2^53, exact in any summation order.  K6 (the score
kernel) is compared on every bin with the oracle's float64 pair terms contracted as two float64 GEMMs, a summation order
different from the kernel's and from orc.s3_scores_f64.  Each reference is pinned to the oracle in the same test.

s3_score_launch restates the score kernel's launch selection and gram_schedule the Gram kernel's tile schedule, so the
CPU-only tests below can show which blocking and which schedule each case reaches.  Inputs are drawn on the device from a
seeded torch.Generator; their pad bytes hold a label no kernel may read.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import epilogos_oracle as orc            # noqa: E402  (checker only)

RTOL, ATOL = 1e-9, 1e-12
PAD = 100                     # pad byte of the label matrices: not a state


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import build, engine
    build.build()
    engine.device_info()
    return engine


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def states(bins, cols, k, seed):
    """Labels [bins, pitch] on the device: each bin keeps one dominant state in about 60 % of its biosamples and draws the
    rest uniformly, and every 97th bin is all state K - 1."""
    g = gen(seed)
    x = torch.full((bins, (cols + 15) & ~15), PAD, dtype=torch.int8, device="cuda")
    step = 1 << 18
    for lo in range(0, bins, step):
        n = min(step, bins - lo)
        dom = torch.randint(0, k, (n, 1), generator=g, device="cuda", dtype=torch.int8)
        other = torch.randint(0, k, (n, cols), generator=g, device="cuda", dtype=torch.int8)
        keep = torch.rand((n, cols), generator=g, device="cuda") < 0.6
        x[lo:lo + n, :cols] = torch.where(keep, dom, other)
    x[::97, :cols] = k - 1
    return x


def one_hot(x, cols, k):
    """float64 [bins, cols*K]: OH[b][i*K + a] = (x[b, i] == a)."""
    return torch.nn.functional.one_hot(x[:, :cols].long(), k).reshape(x.shape[0], cols * k).to(torch.float64)


def zero_diagonal_blocks(t4):
    """t4[i, i] = 0 for every i of a [C, C, ...] tensor (in place)."""
    idx = torch.arange(t4.shape[0], device=t4.device)
    t4[idx, idx] = 0
    return t4


# ------------------------------------------------------------------------------------------------ references
def gram_reference(x, cols, k, chunk=16384):
    """N3 [C, C, K, K] int64: OH^T OH over bin chunks, accumulated in int64, i == j blocks zeroed."""
    ck = cols * k
    g = torch.zeros((ck, ck), dtype=torch.int64, device="cuda")
    for lo in range(0, x.shape[0], chunk):
        oh = one_hot(x[lo:lo + chunk], cols, k)
        g += (oh.T @ oh).to(torch.int64)
        del oh
    n3 = g.view(cols, k, cols, k).permute(0, 2, 1, 3).contiguous()
    del g
    return zero_diagonal_blocks(n3)


def score_reference(x, cols, k, terms, chunk=4096):
    """float64 [bins, K]: with M[(i,a)][(j,c)] = T[i][j][a][c] (i == j blocks zeroed), U = OH M and
    score[b][s] = sum_j OH[b][j*K + s] U[b][j*K + s] -- the terms of the ordered pairs (i, j) of a bin, bucketed by x_j."""
    ck = cols * k
    t = zero_diagonal_blocks(torch.from_numpy(terms).cuda())
    m = t.permute(0, 2, 1, 3).reshape(ck, ck)
    del t
    out = torch.empty((x.shape[0], k), dtype=torch.float64, device="cuda")
    for lo in range(0, x.shape[0], chunk):
        oh = one_hot(x[lo:lo + chunk], cols, k)
        u = torch.where(oh != 0, oh @ m, 0.0)          # an empty bucket sums +0.0 terms, as in the kernel
        out[lo:lo + oh.shape[0]] = u.view(oh.shape[0], cols, k).sum(dim=1)
    return out


def pin_gram_reference(x, cols, k):
    """The Gram reference equals the oracle's N3 on a small corner of the input."""
    small = x[:257, :min(cols, 40)]
    c = small.shape[1]
    assert torch.equal(gram_reference(small, c, k).cpu(), torch.from_numpy(orc.s3_expected_counts(small.cpu().numpy(), k)))


def assert_counts_equal(got, want, k):
    if torch.equal(got, want):
        return
    ne = got != want
    bad = ne.nonzero()[:8].tolist()
    desc = []
    for i, j, a, c in bad:
        m, q = sorted((i * k + a, j * k + c))
        desc.append("[%d,%d,%d,%d] = %d, want %d (Gram row %d, col %d: 256-block %d,%d)"
                    % (i, j, a, c, int(got[i, j, a, c]), int(want[i, j, a, c]), m, q, m // 256, q // 256))
    raise AssertionError("%d of %d counts differ: %s" % (int(ne.sum()), got.numel(), "; ".join(desc)))


def assert_scores_close(got, want, bc):
    got, want = got.cpu().numpy(), want.cpu().numpy()
    bad = ~np.isclose(got, want, rtol=RTOL, atol=ATOL)
    if bad.any():
        b, s = np.nonzero(bad)
        pos = ["bin %d (CTA %d, local %d) state %d: %r, want %r" % (b[n], b[n] // bc, b[n] % bc, s[n], got[b[n], s[n]],
                                                                    want[b[n], s[n]]) for n in range(min(8, len(b)))]
        raise AssertionError("%d of %d scores differ in %d bins: %s" % (bad.sum(), bad.size, len(np.unique(b)),
                                                                     "; ".join(pos)))


# ------------------------------------------------------------------------------------------------ launch restatements
def s3_score_launch(k, bins):
    """(bins per thread, slabs in the ring) that epi_scores_s3 and launch_s3_score (csrc/s3_score.cu) choose, from their
    own constants: 256 consumer threads, j-blocks of JC = 8 biosamples, score rows of K | 1 doubles, the 220 KB fit of the
    rows and two slabs, and the 224 KB budget of the ring."""
    slab = 8 * ((k * k + 1) & ~1) * 8
    rows = lambda bpt: 256 * bpt * (k | 1) * 8          # noqa: E731
    bpt = 4 if bins > 512 else 2 if bins > 256 else 1
    while rows(bpt) + 2 * slab + 256 > 220 * 1024 and bpt > 1:
        bpt //= 2
    assert rows(bpt) + 2 * slab + 256 <= 220 * 1024
    r = (rows(bpt) + 127) & ~127
    return bpt, next(n for n in (4, 3, 2) if n == 2 or r + n * slab + 128 <= 224 * 1024)


def gram_schedule(cols, k, bins, sms=148, chunk=131072):
    """The schedule of epi_s3_plan / epi_s3_gram (csrc/s3_gram.cu) as engine.s3_expected_tiles runs it on a GPU with `sms`
    SMs: 256 x 256 blocks on or above the diagonal of the Gram matrix, rasterised in groups of 8 block columns, computed by
    min(sms / 2, blocks) CTA pairs, one launch per `chunk` bins."""
    nt = -(-cols * k // 256)
    groups = -(-nt // 8)
    blocks = nt * (nt + 1) // 2
    pairs = min(sms // 2, blocks)
    launches = -(-bins // chunk)
    return dict(nt=nt, groups=groups, last_group=nt - 8 * (groups - 1), blocks=blocks, pairs=pairs,
                per_pair=-(-blocks // pairs), launches=launches, last_launch=bins - chunk * (launches - 1))


# (K, C, bins).  Several CTAs with one valid bin in the tail CTA (n * BC + 1) for every blocking but (1, 4), which only
# ever runs as a single CTA; exact multiples of BC; both sides of the bin-count switches; widths at the j-block edges.
SCORE_CASES = [
    (15, 833, 3073),      # (4, 4)
    (18, 833, 4097),      # (4, 3)
    (20, 61, 2049),       # (4, 2)
    (22, 70, 1537),       # (2, 4)
    (25, 97, 1537),       # (2, 3)
    (26, 61, 1025),       # (2, 2)
    (26, 61, 1024),       # (2, 2), two full CTAs
    (29, 50, 769),        # (1, 3)
    (32, 40, 513),        # (1, 2)
    (32, 40, 768),        # (1, 2), three full CTAs
    (18, 33, 200),        # (1, 4)
    (27, 45, 200),        # (1, 3)
    (18, 33, 256), (18, 33, 257), (18, 33, 512), (18, 33, 513),
    (15, 2, 2049), (29, 3, 2049), (18, 7, 2049), (22, 8, 2049), (32, 9, 2049), (25, 16, 2049), (20, 17, 2049),
    (1, 2, 2049), (1, 9, 1025), (2, 3, 2049), (2, 17, 513),
]

# (C, K, bins)
GRAM_CASES = [
    (833, 18, 300_001),   # three launches, the last of 37,857 bins; 24 blocks per CTA pair; a last raster group of 3
    (1422, 18, 20_001),   # 100 block columns in 13 raster groups, 69 blocks per CTA pair
    (400, 25, 50_001),    # 40 block columns: exactly 5 full raster groups
    (300, 32, 50_001),    # 38 block columns
] + [(c, k, b) for c, k in ((16, 16), (8, 32), (17, 16), (9, 32)) for b in (1, 128, 129)]


def test_s3_score_launch_table():
    """The (bins per thread, slabs) blocking by state count: for more than 512 bins 4 bins per thread up to K = 20, 2 up
    to K = 28, then 1; for 257..512 bins 2 up to K = 28, then 1; for 1..256 bins 1.  The ring holds 4 slabs up to K = 17
    / 22 / 26 (4 / 2 / 1 bins per thread), 3 up to K = 19 / 25 / 29, else 2.  JC = 8 fits at every K <= 32."""
    def table(k, bins):
        bpt = 4 if bins > 512 else 2 if bins > 256 else 1
        if bpt == 4 and k > 20:
            bpt = 2
        if bpt == 2 and k > 28:
            bpt = 1
        four, three = {4: (17, 19), 2: (22, 25), 1: (26, 29)}[bpt]
        return bpt, 4 if k <= four else 3 if k <= three else 2
    for k in range(1, 33):
        for bins in (1, 200, 256, 257, 512, 513, 10 ** 7):
            assert s3_score_launch(k, bins) == table(k, bins), (k, bins)
            if bins > 256:
                assert s3_score_launch(k, bins) != (1, 4)             # one bin per thread and 4 slabs: one CTA only


def test_s3_score_cases_reach_every_blocking():
    """Every (bins per thread, slabs) pair is reached, each case runs with a symmetric and a non-symmetric table, and
    every blocking but (1, 4) runs several CTAs with a tail CTA of one valid bin."""
    pairs = {(b, n) for b in (4, 2, 1) for n in (4, 3, 2)}
    assert {s3_score_launch(k, bins) for k, _, bins in SCORE_CASES} == pairs
    tails = set()
    for k, _, bins in SCORE_CASES:
        bpt, nslab = s3_score_launch(k, bins)
        if bins > 256 * bpt and bins % (256 * bpt) == 1:
            tails.add((bpt, nslab))
    assert tails == pairs - {(1, 4)}


def test_s3_gram_cases_reach_their_schedules():
    """The schedules the Gram cases claim, on 148 SMs, and the tile count epi_s3_plan reports (no device needed)."""
    from epilogos_b200 import engine
    s = [gram_schedule(c, k, b) for c, k, b in GRAM_CASES[:4]]
    assert (s[0]["nt"], s[0]["groups"], s[0]["last_group"], s[0]["per_pair"]) == (59, 8, 3, 24)
    assert (s[0]["launches"], s[0]["last_launch"]) == (3, 37857) and s[0]["last_launch"] % 128
    assert (s[1]["nt"], s[1]["groups"], s[1]["last_group"], s[1]["per_pair"]) == (100, 13, 4, 69)
    assert (s[2]["nt"], s[2]["groups"], s[2]["last_group"]) == (40, 5, 8)
    assert (s[3]["nt"], s[3]["groups"], s[3]["last_group"]) == (38, 5, 6)
    for c, k, b in GRAM_CASES:
        sc = gram_schedule(c, k, b)
        assert engine.s3_plan(b, c, k)["ntiles"] == 2 * sc["blocks"]
        if c * k == 256:
            assert sc["blocks"] == 1
        elif c * k < 512:
            assert sc["blocks"] == 3                               # one column into the second block column


# ------------------------------------------------------------------------------------------------ K6 scores
def device_exp(eng, x, cols, k):
    tiles, plan = eng.s3_expected_tiles(x, cols, k)
    return eng.s3_finalize(tiles, cols, k, plan["mp"], x.shape[0], want_counts=False)[1]


def perturbed(exp, seed):
    """A non-symmetric table: every entry scaled by its own factor in [0.5, 1.5), about 2 % of the entries and the whole
    pair block (C - 1, 0) zero (masked terms) while the block (0, C - 1) is not, and non-zero i == j blocks, which no
    kernel may read."""
    g = gen(seed)
    e = exp * (0.5 + torch.rand(exp.shape, generator=g, device="cuda"))
    e[torch.rand(exp.shape, generator=g, device="cuda") < 0.02] = 0
    e[-1, 0] = 0
    e[0, -1] = float(exp.max())
    idx = torch.arange(exp.shape[0], device="cuda")
    e[idx, idx] = torch.rand(e[idx, idx].shape, generator=g, device="cuda") * float(exp.max())
    return e


@pytest.mark.parametrize("sym", [True, False], ids=["sym", "ordered"])
@pytest.mark.parametrize("k,cols,bins", SCORE_CASES)
def test_s3_scores_on_every_bin(eng, k, cols, bins, sym):
    """Every bin of every CTA, float64 output within 1e-9 of the GEMM reference; the float32 output is its rounding, with
    or without a float64 output.  A symmetric table takes the unordered-pair kernel, a non-symmetric one the ordered-pair
    kernel."""
    x = states(bins, cols, k, seed=bins * 64 + k)
    exp = device_exp(eng, x, cols, k)
    if not sym:
        exp = perturbed(exp, seed=cols)
    e = exp.cpu().numpy()
    assert np.array_equal(e, e.transpose(1, 0, 3, 2)) == sym
    t = orc.s3_pair_terms(cols, e, np.float64)
    terms = eng.s3_terms(exp.reshape(-1), cols, k)
    s32, s64 = eng.scores_s3(x, cols, k, terms, want64=True)
    ref = score_reference(x, cols, k, t)
    bc = 256 * s3_score_launch(k, bins)[0]
    # the reference against the oracle on the first and the last bin of every CTA
    ends = sorted({b for lo in range(0, bins, bc) for b in (lo, min(lo + bc, bins) - 1)})
    np.testing.assert_allclose(ref[ends].cpu().numpy(), orc.s3_scores_f64(x[ends, :cols].cpu().numpy(), k, e, terms=t),
                               rtol=RTOL, atol=ATOL)
    assert_scores_close(s64, ref, bc)
    assert torch.equal(s32, s64.to(torch.float32))
    assert torch.equal(eng.scores_s3(x, cols, k, terms), s32)


# ------------------------------------------------------------------------------------------------ K3 + finalize
@pytest.mark.parametrize("cols,k,bins", GRAM_CASES)
def test_s3_gram_and_finalize_on_every_tile(eng, cols, k, bins):
    """The whole [C, C, K, K] count table equals the reference exactly, and the float32 table is the oracle's
    normalisation of it byte for byte."""
    x = states(bins, cols, k, seed=cols * 100 + k)
    tiles, plan = eng.s3_expected_tiles(x, cols, k)
    counts, exp = eng.s3_finalize(tiles, cols, k, plan["mp"], bins)
    del tiles
    ref = gram_reference(x, cols, k)
    assert_counts_equal(counts, ref, k)
    del counts
    assert exp.cpu().numpy().tobytes() == orc.normalize_expected(ref.cpu().numpy()).tobytes()
    pin_gram_reference(x, cols, k)


@pytest.mark.parametrize("cols,k,bins", [(97, 25, 5_001), (17, 16, 1_000)])
def test_s3_gram_one_k_step_per_launch(eng, cols, k, bins):
    """chunk_bins = 128: one k-step per launch, every launch after the first accumulating into the tile buffer.  The tiles
    equal those of the default chunking word for word (compared before epi_s3_finalize writes its tile index behind
    them), and their counts equal the reference."""
    x = states(bins, cols, k, seed=bins + k)
    t0, plan = eng.s3_expected_tiles(x, cols, k)
    t1, _ = eng.s3_expected_tiles(x, cols, k, chunk_bins=128)
    n = plan["ntiles"] * 128 * 256
    assert torch.equal(t0[:n], t1[:n])
    counts, _ = eng.s3_finalize(t1, cols, k, plan["mp"], bins, want_exp=False)
    assert_counts_equal(counts, gram_reference(x, cols, k), k)


# ------------------------------------------------------------------------------------------------ host entry point
def test_s3_host_entry_point_over_two_gram_launches(eng):
    """epi_s3_host with more bins than one Gram launch takes: the float32 table is the normalised reference byte for
    byte; the float32 scores are the rounding of the score reference, but for rare 1-ulp cases."""
    from test_gpu_parity import assert_f32_close
    k, cols, bins = 25, 40, 140_001
    x = states(bins, cols, k, seed=7)
    exp, s32 = eng.s3_host(x.cpu(), cols, k)
    ref = gram_reference(x, cols, k)
    assert exp.tobytes() == orc.normalize_expected(ref.cpu().numpy()).tobytes()
    t = orc.s3_pair_terms(cols, exp, np.float64)
    sref = score_reference(x, cols, k, t).cpu().numpy()
    ends = [0, 131071, 131072, bins - 1]
    np.testing.assert_allclose(sref[ends], orc.s3_scores_f64(x[ends, :cols].cpu().numpy(), k, exp, terms=t), rtol=RTOL,
                               atol=ATOL)
    assert_f32_close(s32, sref.astype(np.float32))
