"""The kernels at the far ends of the ranges their entry points accept, and in the steady state of their persistent loops.

Every reference is exact integer arithmetic or the float64 numpy oracle, never the kernel under test (the group counts are
also compared with gather + K1, which is a different kernel).  Large inputs are drawn on the device from a seeded
torch.Generator.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import epilogos_oracle as orc            # noqa: E402  (checker only)
from oracle import simsearch_oracle as so            # noqa: E402

RTOL, ATOL = 1e-9, 1e-12


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


def u16(cnt):
    """int16 tensor holding uint16 counts -> int64 tensor of the counts."""
    return cnt.to(torch.int64) & 0xffff


def oracle_counts(x, cols, k, block=256):
    """orc.bin_counts of a device state matrix [bins, pitch], a block of rows at a time."""
    return np.concatenate([orc.bin_counts(x[lo:lo + block, :cols].cpu().numpy(), k)
                           for lo in range(0, x.shape[0], block)])


def check_counts_downstream(eng, cnt, width, k):
    """K2, K4, the S1 scores and the S2 scores (TABLE and DIRECT) of the counts `cnt` against the exact int64 tables and
    the float64 oracle; float32 scores must be the rounding of the float64 ones."""
    c = u16(cnt).cpu().numpy()
    n1 = c.sum(axis=0)
    n2 = c.T @ c - np.diag(n1)                        # exact: the products stay below 2^32, the sums below 2^63
    n1t, n2t = eng.expected_tables(cnt, width)
    assert np.array_equal(n1t.cpu().numpy(), n1) and np.array_equal(n2t.cpu().numpy(), n2)
    e1, e2 = eng.normalize(n1t), eng.normalize(n2t)
    assert e1.cpu().numpy().tobytes() == orc.normalize_expected(n1).tobytes()
    assert e2.cpu().numpy().tobytes() == orc.normalize_expected(n2).tobytes()
    ref1 = orc.s1_scores_from_counts(c, width, e1.cpu().numpy(), np.float64)
    ref2 = orc.s2_scores_from_counts(c, width * (width - 1), e2.cpu().numpy(), np.float64)
    for mode in (eng.EPI_SCORE_TABLE, eng.EPI_SCORE_DIRECT):
        s32, s64 = eng.scores_s1(cnt, width, e1, want64=True, mode=mode)
        np.testing.assert_allclose(s64.cpu().numpy(), ref1, rtol=RTOL, atol=ATOL)
        assert torch.equal(s32, s64.to(torch.float32))
        s32, s64 = eng.scores_s2(cnt, width, e2, want64=True, mode=mode)
        np.testing.assert_allclose(s64.cpu().numpy(), ref2, rtol=RTOL, atol=ATOL)
        assert torch.equal(s32, s64.to(torch.float32))


# ------------------------------------------------------------------------------------------------ the widest input
def special_states(k):
    """State 0 and the states that share a 32-bit counter word with it (8, 16, and 17 through the 17/18-state
    separation), where they exist, and the last state."""
    return sorted({s for s in (0, 8, 16, 17, k - 1) if s < k})


@pytest.mark.parametrize("k", [15, 18, 25])
@pytest.mark.parametrize("cols", [65520, 65521, 65528, 65535])
def test_k1_at_the_widest_rows_and_its_counts_downstream(eng, cols, k):
    """K1 pads a row to whole chunks of 16-byte vectors and counts the zero pad in state 0.  At widths 65,521..65,535
    the padded row is longer than 65,535 labels, so a bin with nearly every label in state 0 takes state 0's 16-bit
    counter past its end.  Whole rows of state 0 and of the states that share its counter word catch a carry into the
    neighbouring counter; the counts then go through K2, K4 and the S1 / S2 scores (DIRECT S1 and DFMA-TABLE S2 at these
    widths) with counts of up to 65,535."""
    bins = 3001
    pitch = eng.pitch_for(cols)
    g = gen(cols * 31 + k)
    x = torch.randint(0, k, (bins, pitch), generator=g, device="cuda", dtype=torch.int8)
    x[:, cols:] = 5                                          # pad bytes are never interpreted
    r = 0
    for s in special_states(k):
        x[r, :cols] = s                                      # the whole row in state s
        x[r + 1, :cols] = s
        x[r + 1, cols // 2] = (s + 1) % k                    # all but one label
        x[r + 2, : cols - 32] = s                            # all but the last 32 labels (random)
        r += 3
    skew = torch.rand((500, cols), generator=g, device="cuda") < 0.5
    x[r:r + 500, :cols][skew] = 0                            # about half of each of these rows in state 0
    cnt = eng.bin_counts(x, cols, k)
    got = u16(cnt).cpu().numpy()
    ref = oracle_counts(x, cols, k)
    bad = tuple(np.argwhere(got != ref)[:6].T)
    assert not len(bad[0]), "[bin, state] %s: counts %s, want %s" % (np.transpose(bad).tolist(), got[bad].tolist(),
                                                                    ref[bad].tolist())
    assert got[0, 0] == cols
    check_counts_downstream(eng, cnt, cols, k)


def constructed_rows(width, k, rng):
    """Count rows of one width: every state alone at `width`, the pairs (1, width - 1) and, when width == 65535,
    (32768, 32767) -- products of up to about 2^32 -- then multinomial rows."""
    rows = []
    for s in range(k):
        row = np.zeros(k, np.int64)
        row[s] = width
        rows.append(row)
        row = np.zeros(k, np.int64)
        row[s], row[(s + 1) % k] = 1, width - 1
        rows.append(row)
        if width == 65535:
            row = np.zeros(k, np.int64)
            row[s], row[(s + 7) % k] = 32768, 32767
            rows.append(row)
    rows = np.array(rows)
    rand = rng.multinomial(width, rng.dirichlet(np.ones(k)), size=1000)
    return np.concatenate([rows, rand])


@pytest.mark.parametrize("k", [15, 18, 25])
@pytest.mark.parametrize("width", [32768, 65535])
def test_counts_of_the_widest_widths_downstream(eng, width, k):
    rng = np.random.default_rng(width + k)
    c = constructed_rows(width, k, rng)
    assert c.max() == width and (c.sum(axis=1) == width).all()
    cnt = torch.from_numpy(c.astype(np.uint16).view(np.int16)).cuda()
    check_counts_downstream(eng, cnt, width, k)


# ------------------------------------------------------------------------------------------------ K2 in steady state
@pytest.mark.parametrize("k", [7, 15, 17, 18, 32])
def test_k2_tensor_core_gram_drains_in_mid_run(eng, k):
    """k2_tc_kernel accumulates a CTA's tiles of 128 bins in tensor memory and drains the accumulator after every
    T2_DRAIN = 256 tiles and after its last one; launch_k2_tc runs a persistent grid of 4 CTAs per SM.  With this many
    bins every CTA drains twice in mid-run and once more after a partial window, and the last tile is partial.  One count
    array holds 255 everywhere (every low-byte product saturated), the other uniform uint16 counts.  The reference is exact:
    float64 Gram products over 2^20 bins (65535^2 * 2^20 < 2^53), summed in int64."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ctas, drain, tile = 4 * sms, 256, 128
    bins = ctas * tile * (2 * drain + 37) + 77
    ntiles = -(-bins // tile)
    per_cta = ntiles // ctas
    assert per_cta >= 2 * drain + 1 and per_cta % drain != 0 and bins % tile != 0
    g = gen(k)
    arrays = (lambda: torch.full((bins, k), 255, dtype=torch.int16, device="cuda"),
              lambda: torch.randint(-32768, 32768, (bins, k), generator=g, device="cuda", dtype=torch.int16))
    for make in arrays:
        cnt = make()
        n1 = torch.zeros(k, dtype=torch.int64, device="cuda")
        n2 = torch.zeros((k, k), dtype=torch.int64, device="cuda")
        for lo in range(0, bins, 1 << 20):
            c = u16(cnt[lo:lo + (1 << 20)])
            n1 += c.sum(dim=0)
            cf = c.to(torch.float64)
            n2 += (cf.T @ cf).to(torch.int64)
            del c, cf
        n2 -= torch.diag(n1)
        n1t, n2t = eng.expected_tables(cnt, 65535)
        assert torch.equal(n1t, n1) and torch.equal(n2t, n2)
        del cnt
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ column groups
GROUP_LIMIT = 65520          # the most columns a group may list: whole chunks of 48 (16) labels below 65,536


def eight_groups(cols, rng):
    """All columns (up to the group limit), two disjoint halves, two overlapping ranges, two scattered subsets, one
    column."""
    half = cols // 2
    return [np.arange(min(cols, GROUP_LIMIT)), np.arange(half), np.arange(half, cols),
            np.arange(cols // 4, cols // 4 + cols // 3), np.arange(cols // 3, cols - 1),
            np.sort(rng.choice(cols, size=cols // 5, replace=False)),
            rng.choice(cols, size=min(cols - 3, GROUP_LIMIT), replace=False),        # unsorted
            np.array([cols - 1])]


@pytest.mark.parametrize("k", [15, 18, 25])
@pytest.mark.parametrize("bins,cols", [(2_000_001, 833), (300_001, 2100), (3_001, 65535)])
def test_group_counts_in_steady_state(eng, bins, cols, k):
    """Enough bins for at least 5 tiles per CTA: the staged tile is reused across iterations, at 2,100 columns a tile
    holds fewer than 128 rows, at 65,535 columns about 3, and mid-array warps store to destinations that are not 16-byte
    aligned.  Bit-equal to gather + K1 per group, and to numpy on a sample of 2,000 bins."""
    rng = np.random.default_rng(bins + cols + k)
    g = gen(bins + k)
    x = torch.randint(0, k, (bins, eng.pitch_for(cols)), generator=g, device="cuda", dtype=torch.int8)
    x[: bins // 7] = k - 1                                                      # long runs of one state
    x[bins // 7: bins // 7 + 50] = 0
    groups = eight_groups(cols, rng)
    got = eng.group_counts(x, cols, k, groups)
    assert got.shape == (len(groups), bins, k)
    for i, cols_g in enumerate(groups):
        sub = eng.gather_columns(x, cols, cols_g)
        assert torch.equal(got[i], eng.bin_counts(sub, len(cols_g), k)), i
        del sub
    sample = np.sort(rng.choice(bins, size=2000, replace=False))
    sample[:2] = [0, bins - 1]
    xs = x[torch.from_numpy(sample).cuda(), :cols].cpu().numpy()
    gs = u16(got[:, torch.from_numpy(sample).cuda()]).cpu().numpy()
    for i, cols_g in enumerate(groups):
        assert np.array_equal(gs[i], orc.bin_counts(xs[:, cols_g], k)), i


@pytest.mark.parametrize("k", [15, 18, 25])
def test_group_counts_at_the_group_size_limit(eng, k):
    """The largest group epi_group_counts admits counts rows of one state exactly; one column more is refused."""
    from epilogos_b200._lib import EpilogosB200Error
    cols = 65535
    states = special_states(k)
    x = torch.zeros((len(states), eng.pitch_for(cols)), dtype=torch.int8, device="cuda")
    for r, s in enumerate(states):
        x[r, :cols] = s
    got = u16(eng.group_counts(x, cols, k, [np.arange(GROUP_LIMIT), np.arange(cols - GROUP_LIMIT, cols)]))
    want = torch.zeros((len(states), k), dtype=torch.int64, device="cuda")
    want[torch.arange(len(states)), torch.tensor(states)] = GROUP_LIMIT
    assert torch.equal(got[0], want) and torch.equal(got[1], want)
    with pytest.raises(EpilogosB200Error, match="at most %d fit" % GROUP_LIMIT):
        eng.group_counts(x, cols, k, [np.arange(GROUP_LIMIT + 1)])


# ------------------------------------------------------------------------------------------------ S1 launch dispatch
def s1_launch(k, width):
    """The kernel launch_s1 (csrc/scores.cu) chooses for TABLE mode, from its own constants: K5_WARPS = 8 warps of a
    256-thread CTA, S1_SMEM_TABLE_BYTES = 96 KB, S1_TABLE_MAX_WIDTH = 4095, and the 220 / 226 KB budgets of one SM."""
    if width > 4095:
        return "direct"
    base = 8 * 32 * k * 8 + 8 * 16
    table = k * (width + 1) * 4
    big = 32 * 32 * k * 8 + 32 * 16                 # 1024-thread CTA
    if table <= 96 * 1024 and 4 * (base + table + 1024) > 220 * 1024 and big + table + 1024 <= 226 * 1024:
        return "smem, 1024 threads"
    if table <= 96 * 1024:
        return "smem, 256 threads x %d per SM" % max(1, min(4, 220 * 1024 // (base + table + 1024)))
    return "global table"


def s1_switch_widths(k):
    """Width 1 and both sides of every switch of s1_launch."""
    out = {1}
    for w in range(2, 4097):
        if s1_launch(k, w) != s1_launch(k, w - 1):
            out |= {w - 1, w}
    return sorted(out)


S1_CASES = [(k, w) for k in (2, 7, 15, 18, 25, 32) for w in s1_switch_widths(k)]


def test_s1_switch_widths_cover_every_launch():
    assert s1_switch_widths(18) == [1, 253, 254, 1143, 1144, 1364, 1365, 4095, 4096]
    assert {s1_launch(k, w) for k, w in S1_CASES} == {
        "direct", "global table", "smem, 1024 threads", "smem, 256 threads x 1 per SM", "smem, 256 threads x 2 per SM",
        "smem, 256 threads x 3 per SM", "smem, 256 threads x 4 per SM"}


@pytest.mark.parametrize("k,width", S1_CASES)
def test_s1_scores_on_both_sides_of_every_launch_switch(eng, k, width):
    """TABLE and DIRECT both evaluate kl_direct(c / width, E[s]), so they agree bit for bit; against the oracle within the
    score tolerance.  Multinomial rows plus the extreme counts 0, 1, width - 1 and width of every state."""
    rng = np.random.default_rng(k * 10000 + width)
    c = rng.multinomial(width, rng.dirichlet(np.ones(k) * 0.5), size=5000)
    for s in range(k):
        c[s] = 0
        c[s, s] = width
        c[k + s] = 0
        c[k + s, s], c[k + s, (s + 1) % k] = 1, width - 1
    e1 = rng.dirichlet(np.ones(k)).astype(np.float32)
    cnt = torch.from_numpy(c.astype(np.uint16).view(np.int16)).cuda()
    e1d = torch.from_numpy(e1).cuda()
    t32, t64 = eng.scores_s1(cnt, width, e1d, want64=True, mode=eng.EPI_SCORE_TABLE)
    d32, d64 = eng.scores_s1(cnt, width, e1d, want64=True, mode=eng.EPI_SCORE_DIRECT)
    assert torch.equal(t64, d64) and torch.equal(t32, d32), s1_launch(k, width)
    assert torch.equal(t32, t64.to(torch.float32))
    np.testing.assert_allclose(t64.cpu().numpy(), orc.s1_scores_from_counts(c, width, e1, np.float64), rtol=RTOL,
                               atol=ATOL)


# ------------------------------------------------------------------------------------------------ shuffle and search limits
@pytest.mark.parametrize("c1,c2,ok", [(6399, 6399, True), (6400, 6399, False)])
def test_shuffle_kernel_at_its_shared_memory_limit(eng, c1, c2, ok):
    """The shuffle kernel keeps (2 width + 3) doubles in shared memory, at most 200 KB: 12,798 combined biosamples."""
    from epilogos_b200._lib import EpilogosB200Error
    k, bins = 18, 1000
    rng = np.random.default_rng(c1 + c2)
    p = rng.dirichlet(np.ones(k) * 0.3, size=bins)
    a = np.stack([rng.multinomial(c1, q) for q in p])
    b = np.stack([rng.multinomial(c2, q) for q in p])
    a[0], b[0] = 0, 0
    a[0, 0], b[0, k - 1] = c1, c2
    ca = torch.from_numpy(a.astype(np.int16)).cuda()
    cb = torch.from_numpy(b.astype(np.int16)).cuda()
    if not ok:
        with pytest.raises(EpilogosB200Error, match="too many combined biosamples"):
            eng.shuffled_counts_philox(ca, cb, c1, c2, 3, nperm=2, width=c1 + c2)
        return
    oa, ob = eng.shuffled_counts_philox(ca, cb, c1, c2, 3, nperm=2, width=c1 + c2)
    oa, ob = u16(oa), u16(ob)
    assert bool((oa.sum(dim=2) == c1).all()) and bool((ob.sum(dim=2) == c2).all())
    assert torch.equal(oa + ob, (u16(ca) + u16(cb)).expand(2, bins, k))
    assert not torch.equal(oa[0], oa[1])


def test_similarity_search_at_its_largest_window(eng):
    """K = 64 states and nS = 32 reduced bins, 11 ROIs (one full batch of 8 and a partial one): the distances against the
    restatement of sklearn's formula, the mode against scipy's rule on a genome with repeated windows; K = 65 and nS = 33
    are refused."""
    from epilogos_b200 import similaritySearch_calc as ssc
    from epilogos_b200._lib import EpilogosB200Error
    K, nS, G = 64, 32, 3000
    rng = np.random.default_rng(64)
    genome = rng.random((G, K))
    genome[: G // 2] = np.tile(rng.random((37, K)), (G // 74 + 1, 1))[: G // 2]      # windows that repeat every 37 bins
    starts = [0, 5, 36, 37, 700, 1480, 1600, 2000, 2500, G - nS, 1234]
    rois = np.stack([genome[s:s + nS] for s in starts])
    rois[-1] = rng.random((nS, K))
    gd = torch.from_numpy(genome).cuda()
    dist = ssc.window_distances(gd, ssc.row_norms(gd), torch.from_numpy(rois).cuda())
    assert dist.shape == (len(starts), G - nS + 1)
    d = dist.cpu().numpy()
    for r in range(len(starts)):
        ref = so.window_distances(genome, rois[r])
        # a window's terms are differences of sums of squares of order K: the error of either evaluation is absolute
        np.testing.assert_allclose(d[r], ref, rtol=1e-12, atol=1e-12 * np.median(ref))
    modes = ssc.mode_of_sorted(torch.sort(dist, dim=1).values).cpu().numpy()
    for r in range(len(starts)):
        assert modes[r] == so.float_mode(d[r])
    xx = torch.zeros(G, dtype=torch.float64, device="cuda")
    for k, ns in ((K + 1, nS), (K, nS + 1)):
        with pytest.raises(EpilogosB200Error, match="bad window shape"):
            ssc.window_distances(torch.zeros((G, k), dtype=torch.float64, device="cuda"), xx,
                                 torch.zeros((1, ns, k), dtype=torch.float64, device="cuda"))
