"""GPU parity: the CUDA path (through the C ABI) against the oracle and the reference goldens.

Bit-exact for counts, integer tables and the float32 expected payload.  Scores: float64 output within
1e-9 relative + 1e-12 absolute of the numpy float64 restatement (BASELINE.json north_star tolerance);
float32 output equal to the reference's float32 except for <= 1-ulp rounding-boundary cases.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import epilogos_oracle as orc            # noqa: E402  (checker only)

RTOL, ATOL = 1e-9, 1e-12


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import build, engine
    build.build()
    engine.device_info()
    return engine


def dev_states(eng, x):
    return eng.pack_states(x).cuda()


def gpu_counts(eng, x, k):
    return eng.counts_to_numpy(eng.bin_counts(dev_states(eng, x), x.shape[1], k))


def assert_f32_close(got32, ref32, max_ulp_frac=2e-3):
    """float32 results equal except rounding-boundary cases (at most 1 ulp apart, and rare)."""
    got32 = np.asarray(got32); ref32 = np.asarray(ref32)
    # zeros must carry the reference's sign ("-0.00000" vs "0.00000" in the text output)
    assert np.array_equal(np.signbit(got32[ref32 == 0]), np.signbit(ref32[ref32 == 0]))
    neq = got32 != ref32
    if neq.any():
        a = got32[neq].astype(np.float64); b = ref32[neq].astype(np.float64)
        ulp = np.spacing(np.maximum(np.abs(a), np.abs(b)).astype(np.float32)).astype(np.float64)
        assert np.all(np.abs(a - b) <= ulp * 1.0000001), "float32 scores differ by more than 1 ulp"
        assert neq.mean() <= max_ulp_frac, "too many 1-ulp differences: %g" % neq.mean()


# ------------------------------------------------------------------------------------------------ K1
@pytest.mark.parametrize("bins,cols,k", [
    (1, 1, 2), (5, 15, 3), (31, 16, 15), (33, 17, 16), (127, 48, 17), (129, 49, 18), (300, 143, 18),
    (257, 144, 18), (1000, 145, 25), (700, 833, 18), (515, 833, 15), (260, 127, 15), (130, 1000, 18),
    (140, 2100, 18), (150, 1700, 16), (135, 1100, 32), (4096, 10, 18), (10000, 833, 18),
    # rows of 97..128 bytes: the one-box, 128-byte-swizzled variant of the count kernel (two-bit modes only)
    (300, 128, 16), (500, 100, 18), (77, 113, 15), (1000, 120, 17), (129, 97, 2), (5000, 127, 15), (333, 128, 25),
])
def test_bin_counts_match_oracle(eng, bins, cols, k):
    rng = np.random.default_rng(bins * 7919 + cols * 31 + k)
    x = rng.integers(0, k, size=(bins, cols)).astype(np.int8)
    x[rng.random(bins) < 0.3] = k - 1                         # whole rows of the last state
    got = gpu_counts(eng, x, k)
    ref = orc.bin_counts(x, k)
    assert got.dtype == np.uint16 and got.shape == (bins, k)
    assert np.array_equal(got.astype(np.int64), ref)


def test_bin_counts_any_pitch_and_alignment(eng):
    rng = np.random.default_rng(5)
    x = rng.integers(0, 18, size=(777, 833)).astype(np.int8)
    dense = torch.from_numpy(x).cuda()                        # pitch == cols == 833: repacked on the device
    got = eng.counts_to_numpy(eng.bin_counts(dense, 833, 18))
    assert np.array_equal(got.astype(np.int64), orc.bin_counts(x, 18))
    wide = torch.full((777, 1024), 7, dtype=torch.int8, device="cuda")   # garbage in the pad columns
    wide[:, :833] = dense
    got = eng.counts_to_numpy(eng.bin_counts(wide, 833, 18))
    assert np.array_equal(got.astype(np.int64), orc.bin_counts(x, 18))


def test_bin_counts_empty(eng):
    out = eng.bin_counts(torch.zeros((0, 848), dtype=torch.int8, device="cuda"), 833, 18)
    assert out.shape == (0, 18)


def test_bad_arguments_raise(eng):
    from epilogos_b200._lib import EpilogosB200Error
    x = torch.zeros((4, 16), dtype=torch.int8, device="cuda")
    with pytest.raises(EpilogosB200Error):
        eng.bin_counts(x, 16, 33)
    with pytest.raises(EpilogosB200Error):
        eng.bin_counts(x, 17, 18)


@pytest.mark.parametrize("bins,cols,k", [(1, 1, 2), (37, 833, 18), (1000, 127, 15), (4097, 833, 18), (300, 8, 16),
                                         (129, 17, 32), (515, 1000, 25)])
def test_packed_transport_layout_round_trip(eng, bins, cols, k):
    """Bit-packed transport layout: device pack == host pack; device unpack restores every label; counts of the unpacked
    matrix equal the oracle's (the pad bytes the unpack kernel leaves unwritten are never interpreted)."""
    rng = np.random.default_rng(bins + cols)
    x = rng.integers(0, k, size=(bins, cols)).astype(np.int8)
    xh = eng.pack_states(x, pin=False)
    host_packed, bits = eng.pack_bits_host(xh, cols, k)
    dev_packed, bits2 = eng.pack_bits(xh.cuda(), cols, k)
    assert bits == bits2 and torch.equal(dev_packed.cpu(), host_packed.cpu())
    back = eng.unpack_bits(host_packed.cuda(), cols, bits)
    assert torch.equal(back[:, :cols].cpu(), torch.from_numpy(x))
    got = eng.counts_to_numpy(eng.bin_counts(back, cols, k))
    assert np.array_equal(got.astype(np.int64), orc.bin_counts(x, k))


@pytest.mark.parametrize("cols,k,saliency", [(833, 18, 2), (833, 18, 1), (127, 15, 2)])
def test_single_host_packed_equals_single_host(eng, cols, k, saliency):
    """epi_single_host_packed (packed chunks over PCIe, expanded on the device) == epi_single_host, bit for bit, over
    several H2D chunks."""
    x = orc.synth_states(600_000 if cols < 200 else 300_000, cols, k, seed=3)
    xh = eng.pack_states(x)
    packed, bits = eng.pack_bits_host(xh, cols, k)
    c0, e0, s0 = eng.single_host(xh, cols, k, saliency)
    s0 = s0.copy()
    c1, e1, s1 = eng.single_host_packed(packed, cols, k, saliency, bits)
    assert np.array_equal(c0, c1) and e0.tobytes() == e1.tobytes() and s0.tobytes() == s1.tobytes()
    ref = orc.s1_expected_counts(x, k) if saliency == 1 else orc.s2_expected_counts(x, k)
    assert np.array_equal(c1, ref)


def test_s3_and_paired_host_entry_points(eng, golden):
    """epi_s3_host / epi_paired_host (host matrices in, host results out) against the reference goldens."""
    g = golden("synth_s3_c40_k18")
    x, k = g["x"], int(g["num_states"])
    exp, scores = eng.s3_host(eng.pack_states(x), x.shape[1], k)
    assert exp.tobytes() == g["s3_exp"].tobytes()
    assert np.max(np.abs(scores - g["s3_scores"])) < 2e-2
    np.testing.assert_allclose(scores, orc.s3_scores_f64(x, k, g["s3_exp"]).astype(np.float32), rtol=1e-5, atol=1e-6)
    for name in ("paired_synth_c30_c25_k18", "paired_synth_g20_k18"):
        g = golden(name)
        xa, xb, k, gs, q = g["xa"], g["xb"], int(g["num_states"]), int(g["group_size"]), int(g["quiescent_state"])
        for s in (1, 2):
            r = eng.paired_host(eng.pack_states(xa), xa.shape[1], eng.pack_states(xb), xb.shape[1], k, s, q, group_size=gs,
                                seed=5, nperm=3)
            assert np.array_equal(r["counts"], g["s%d_counts" % s]) and r["exp"].tobytes() == g["s%d_exp" % s].tobytes()
            assert np.array_equal(r["quiescent"], g["s%d_quiescence" % s])
            perm = orc.reference_shuffle_indices(int(g["seed"]), xa.shape[0], xa.shape[1] + xb.shape[1])
            ref = orc.paired_scores(xa, xb, perm, k, s, g["s%d_exp" % s], q, gs)
            if s == 1:
                assert r["delta"].tobytes() == ref["delta"].tobytes()         # exact value table
            else:                                                             # TABLE mode: rare 1-ulp differences of a score
                np.testing.assert_allclose(r["delta"], ref["delta"], rtol=0, atol=2e-7)
                assert (r["delta"] == ref["delta"]).mean() > 0.995
            assert r["null"].shape == (3, xa.shape[0]) and np.isfinite(r["null"]).all()
            assert not np.array_equal(r["null"][0], r["null"][1])
            # same distribution as the replayed reference shuffle (coarse: medians and spread)
            assert abs(np.median(r["null"]) - np.median(ref["null_distances"])) < 0.5 * np.std(ref["null_distances"])


# ------------------------------------------------------------------------------------ K2 / K4 / K5
SINGLE = ["real10_chr1_k18", "real10_chr1_k18_nproc3", "synth_c833_k18", "synth_uniform_c833_k18", "synth_c127_k15"]


@pytest.mark.parametrize("name", SINGLE)
def test_tables_and_scores_match_reference_goldens(eng, golden, name):
    g = golden(name)
    x, k = g["x"], int(g["num_states"])
    c = x.shape[1]
    cnt = eng.bin_counts(dev_states(eng, x), c, k)
    n1, n2 = eng.expected_tables(cnt, c)
    assert np.array_equal(n1.cpu().numpy(), g["s1_counts"])
    assert np.array_equal(n2.cpu().numpy(), g["s2_counts"])
    e1, e2 = eng.normalize(n1), eng.normalize(n2)
    assert e1.cpu().numpy().tobytes() == g["s1_exp"].tobytes()
    assert e2.cpu().numpy().tobytes() == g["s2_exp"].tobytes()
    ref1_64 = orc.s1_scores(x, k, g["s1_exp"], dtype=np.float64)
    ref2_64 = orc.s2_scores(x, k, g["s2_exp"], dtype=np.float64)
    for mode in (eng.EPI_SCORE_TABLE, eng.EPI_SCORE_DIRECT):
        s1_32, s1_64 = eng.scores_s1(cnt, c, e1, want64=True, mode=mode)
        s2_32, s2_64 = eng.scores_s2(cnt, c, e2, want64=True, mode=mode)
        np.testing.assert_allclose(s1_64.cpu().numpy(), ref1_64, rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(s2_64.cpu().numpy(), ref2_64, rtol=RTOL, atol=ATOL)
        assert_f32_close(s1_32.cpu().numpy(), g["s1_scores"])
        assert_f32_close(s2_32.cpu().numpy(), g["s2_scores"])


@pytest.mark.parametrize("k,cols", [(25, 60), (32, 200), (16, 90), (17, 300), (3, 2)])
def test_other_state_models(eng, k, cols):
    rng = np.random.default_rng(k * 100 + cols)
    x = rng.integers(0, k, size=(900, cols)).astype(np.int8)
    cnt = eng.bin_counts(dev_states(eng, x), cols, k)
    n1, n2 = eng.expected_tables(cnt, cols)
    assert np.array_equal(n1.cpu().numpy(), orc.s1_expected_counts(x, k))
    assert np.array_equal(n2.cpu().numpy(), orc.s2_expected_counts(x, k))
    e1, e2 = eng.normalize(n1), eng.normalize(n2)
    assert e1.cpu().numpy().tobytes() == orc.normalize_expected(n1.cpu().numpy()).tobytes()
    assert e2.cpu().numpy().tobytes() == orc.normalize_expected(n2.cpu().numpy()).tobytes()
    for mode in (eng.EPI_SCORE_TABLE, eng.EPI_SCORE_DIRECT):
        _, s1_64 = eng.scores_s1(cnt, cols, e1, want64=True, mode=mode)
        _, s2_64 = eng.scores_s2(cnt, cols, e2, want64=True, mode=mode)
        np.testing.assert_allclose(s1_64.cpu().numpy(), orc.s1_scores(x, k, e1.cpu().numpy(), np.float64),
                                   rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(s2_64.cpu().numpy(), orc.s2_scores(x, k, e2.cpu().numpy(), np.float64),
                                   rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("bins,cols,k", [
    (1, 2, 1), (127, 255, 18), (128, 256, 18), (129, 257, 15), (256, 1023, 7), (300, 2047, 18), (300, 2048, 18),
    (4097, 5000, 4), (640, 65, 31), (33_000, 70, 32), (1000, 833, 2)])
def test_tensor_core_tables_and_scores_edge_shapes(eng, bins, cols, k):
    """K2 / K5-S2 on the tensor cores at the edges of their tiling: fewer bins than one 128-bin tile, exact tile
    multiples, counts that do / do not need the high byte (255 / 256 biosamples), the widest table-driven width (2047) and
    the first width that takes the per-bin path (2048), 258 tiles (33 000 bins, one tile per CTA), odd state counts.
    Accumulator drains in mid-run need far more bins: test_limits_gpu.py."""
    rng = np.random.default_rng(bins * 7 + cols * 3 + k)
    x = rng.integers(0, k, size=(bins, cols)).astype(np.int8)
    if bins > 2:
        x[1, :] = k - 1                      # a bin with a single state: count = cols (largest possible count)
    cnt = eng.bin_counts(dev_states(eng, x), cols, k)
    n1, n2 = eng.expected_tables(cnt, cols)
    assert np.array_equal(n1.cpu().numpy(), orc.s1_expected_counts(x, k))
    assert np.array_equal(n2.cpu().numpy(), orc.s2_expected_counts(x, k))
    n2h = n2.cpu().numpy().copy()
    n2h[n2h == 0] = 1                        # a table without zeros keeps the tensor-core path (zeros -> DIRECT, tested above)
    e2 = orc.normalize_expected(n2h)
    s32, s64 = eng.scores_s2(cnt, cols, torch.from_numpy(e2).cuda(), want64=True)
    ref = orc.s2_scores(x, k, e2, np.float64)
    np.testing.assert_allclose(s64.cpu().numpy(), ref, rtol=RTOL, atol=ATOL)
    assert np.array_equal(s32.cpu().numpy(), s64.cpu().numpy().astype(np.float32))
    e1 = orc.normalize_expected(orc.s1_expected_counts(x, k))
    t32, t64 = eng.scores_s1(cnt, cols, torch.from_numpy(e1).cuda(), want64=True)
    ref1 = orc.s1_scores(x, k, e1, np.float64)
    np.testing.assert_allclose(t64.cpu().numpy(), ref1, rtol=RTOL, atol=ATOL)
    assert_f32_close(t32.cpu().numpy(), ref1.astype(np.float32), max_ulp_frac=1e-4)


@pytest.mark.parametrize("bins,cols,k,kind", [(4_200_000, 833, 18, "realistic"), (2_000_000, 127, 15, "realistic"),
                                              (300_000, 833, 18, "uniform"), (70_000, 200, 32, "uniform"),
                                              (9_000_000, 127, 15, "realistic"), (200_000, 2100, 18, "realistic")])
def test_s2_tables_and_scores_against_independent_references(eng, bins, cols, k, kind):
    """At sizes that run many tiles per CTA, several accumulator drains and every warpgroup slot: the expected tables must
    equal int64 sums over the device counts computed on the host, bit for bit, and the TABLE scores must agree with the
    term-by-term DIRECT evaluation within the score tolerance, with a float32 output that is the rounding of the float64
    one.  9 M x 127 x 15 is the shape that once exposed a race in the release of the count slabs; at width 2100 the TABLE
    scores come from the DFMA kernel instead of the tensor cores."""
    from epilogos_b200 import synth
    x = synth.synth_states_device(bins, cols, k, seed=bins % 97, kind=kind)
    cnt = eng.bin_counts(x, cols, k)
    del x
    c = eng.counts_to_numpy(cnt)
    n1 = c.sum(axis=0, dtype=np.int64)
    n2 = -np.diag(n1)
    for lo in range(0, bins, 1 << 21):
        ct = np.ascontiguousarray(c[lo:lo + (1 << 21)].T, dtype=np.int64)     # state-major rows: a fast integer product
        n2 += ct @ ct.T
    del c, ct
    n1t, n2t = eng.expected_tables(cnt, cols)
    assert np.array_equal(n1t.cpu().numpy(), n1) and np.array_equal(n2t.cpu().numpy(), n2)
    assert int(n1t.sum()) == bins * cols and int(n2t.sum()) == bins * cols * (cols - 1)
    assert bool((n2t > 0).all())                  # no zero in the expected table: TABLE mode does not fall back to DIRECT
    e2 = eng.normalize(n2t)
    _, ref64 = eng.scores_s2(cnt, cols, e2, want64=True, mode=eng.EPI_SCORE_DIRECT)
    s32, s64 = eng.scores_s2(cnt, cols, e2, want64=True, mode=eng.EPI_SCORE_TABLE)
    assert bool(((ref64 - s64).abs() <= RTOL * ref64.abs() + ATOL).all())
    assert torch.equal(s32, s64.to(torch.float32))


def test_foreign_expected_table_with_zeros_is_masked(eng):
    """klScoreND masks terms whose expected frequency is 0 (scores.py:550); a table computed from other
    data can have zeros where this data has observations."""
    rng = np.random.default_rng(77)
    k, cols = 18, 50
    x = rng.integers(0, k, size=(400, cols)).astype(np.int8)
    e1 = orc.normalize_expected(orc.s1_expected_counts(x, k)).copy()
    e2 = orc.normalize_expected(orc.s2_expected_counts(x, k)).copy()
    e1[[2, 9]] = 0
    e2[3, :] = 0; e2[:, 11] = 0; e2[5, 5] = 0
    cnt = eng.bin_counts(dev_states(eng, x), cols, k)
    _, s1 = eng.scores_s1(cnt, cols, torch.from_numpy(e1).cuda(), want64=True)
    _, s2 = eng.scores_s2(cnt, cols, torch.from_numpy(e2).cuda(), want64=True)
    np.testing.assert_allclose(s1.cpu().numpy(), orc.s1_scores(x, k, e1, np.float64), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(s2.cpu().numpy(), orc.s2_scores(x, k, e2, np.float64), rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("name,sal", [("real10_chr1_k18", 1), ("real10_chr1_k18", 2), ("synth_c833_k18", 2),
                                      ("synth_c127_k15", 1), ("synth_c127_k15", 2)])
def test_single_host_entry_point(eng, golden, name, sal):
    g = golden(name)
    x, k = g["x"], int(g["num_states"])
    counts, exp, scores = eng.single_host(np.ascontiguousarray(x), x.shape[1], k, sal)   # dense pitch, pageable
    assert np.array_equal(counts, g["s%d_counts" % sal])
    assert exp.tobytes() == g["s%d_exp" % sal].tobytes()
    assert_f32_close(scores, g["s%d_scores" % sal])
    counts2, exp2, scores2 = eng.single_host(eng.pack_states(x), x.shape[1], k, sal)      # pinned, padded pitch
    assert np.array_equal(counts2, counts) and exp2.tobytes() == exp.tobytes()
    assert np.array_equal(scores2, scores)


# ---------------------------------------------------------------- BASELINE configs[0] (substitute): real chr1
def test_full_real_chr1_against_reference(eng, golden):
    """All 1,246,253 bins of the real chr1 matrix (10 biosamples, 18 states) through the host-buffer entry point: tables
    and exp_freq payload bit-exact against the reference run, float32 scores against the oracle (itself pinned to the
    reference's sha256 digests in test_oracle_golden.py), and the reference's own top-100 regions of interest from the
    GPU scores: identical regions in identical order."""
    from epilogos_b200 import roi
    g = golden("real10_chr1_full")
    x, k = g["x"], int(g["num_states"])
    scores = {}
    for sal in (1, 2):
        counts, exp, sc = eng.single_host(eng.pack_states(x), x.shape[1], k, sal)
        assert np.array_equal(counts, g["s%d_counts" % sal])
        assert exp.tobytes() == g["s%d_exp" % sal].tobytes()
        ref = orc.s1_scores(x, k, exp) if sal == 1 else orc.s2_scores(x, k, exp)
        assert_f32_close(sc, ref)
        assert_f32_close(sc[:2000], g["s%d_scores_head" % sal])
        scores[sal] = sc.copy()          # single_host reuses one pinned result buffer per shape
    starts = np.arange(len(x), dtype=np.int64) * 200
    sel = roi.max_mean(starts, starts + 200, scores[1].sum(axis=1), 50, 100)
    assert np.array_equal(sel["original_idx"], g["roi_original_idx"])
    assert np.array_equal(sel["start"], g["roi_start"]) and np.array_equal(sel["end"], g["roi_end"])
    # S2: same regions, same order as the selection made from the oracle's scores
    ref2 = orc.s2_scores(x, k, g["s2_exp"])
    want = roi.max_mean(starts, starts + 200, ref2.sum(axis=1), 50, 100)
    got = roi.max_mean(starts, starts + 200, scores[2].sum(axis=1), 50, 100)
    assert np.array_equal(got["original_idx"], want["original_idx"])


def test_wide_833_roi_rankings_against_reference(eng, golden):
    """Downstream parity target at the benchmark width (833 biosamples x 18 states, 24,000 bins): the top-100 regions of
    interest computed from the CUDA scores equal the ranking the UNMODIFIED reference produced with its own
    helpers.maxMean on its own scores -- identical regions in identical order, for S1 and for S2 (tensor-core TABLE
    evaluation); S2 also on the real-data slice.  S3 (160 bins): the reference accumulates in float32 (its scores carry
    ~1e-3 of noise), so the CUDA ranking is held to the one from the float64 restatement and its overlap with the
    reference's regions is reported."""
    import hashlib
    from epilogos_b200 import roi
    g = golden("roi_wide_c833_k18")
    bins, cols, k = int(g["bins"]), int(g["cols"]), int(g["num_states"])
    x = orc.synth_states(bins, cols, k, int(g["seed"]))
    assert hashlib.sha256(np.ascontiguousarray(x).tobytes()).digest() == g["x_sha256"].tobytes()
    starts = np.arange(bins, dtype=np.int64) * 200
    xh = eng.pack_states(x)
    for sal in (1, 2):
        tag = "s%d" % sal
        counts, exp, sc = eng.single_host(xh, cols, k, sal)
        assert exp.tobytes() == g[tag + "_exp"].tobytes()
        sel = roi.max_mean(starts, starts + 200, sc.sum(axis=1), 50, 100)
        assert np.array_equal(sel["original_idx"], g[tag + "_roi_original_idx"]), "S%d ranking differs" % sal
        assert np.array_equal(sel["start"], g[tag + "_roi_start"]) and np.array_equal(sel["end"], g[tag + "_roi_end"])
    # S2 on real data (10 biosamples): the reference's ranking
    real = golden("real10_chr1_k18")["x"]
    counts, exp, sc = eng.single_host(eng.pack_states(real), real.shape[1], 18, 2)
    assert exp.tobytes() == g["real_s2_exp"].tobytes()
    rs = np.arange(len(real), dtype=np.int64) * 200
    sel = roi.max_mean(rs, rs + 200, sc.sum(axis=1), 50, 100)
    assert np.array_equal(sel["original_idx"], g["real_s2_roi_original_idx"])
    # S3
    x3 = x[:160]
    e3, s3 = eng.s3_host(eng.pack_states(x3), cols, k)
    ref64 = orc.s3_scores_f64(x3, k, e3).astype(np.float32)
    s3s = np.arange(160, dtype=np.int64) * 200
    got = roi.max_mean(s3s, s3s + 200, s3.sum(axis=1), 5, 100)
    want = roi.max_mean(s3s, s3s + 200, ref64.sum(axis=1), 5, 100)
    assert np.array_equal(got["original_idx"], want["original_idx"])
    assert np.max(np.abs(s3 - g["s3_scores"])) < 2e-2
    common = len(set(got["original_idx"].tolist()) & set(g["s3_roi_original_idx"].tolist()))
    print("S3 regions shared with the reference's float32 ranking: %d of %d" % (common, len(g["s3_roi_original_idx"])))


# -------------------------------------------------------------------------------- full-size properties
def test_whole_genome_shape_properties(eng):
    """BASELINE configs[1] at full size (15.5 M bins x 833 biosamples x 18 states): size-independent invariants."""
    from epilogos_b200 import synth
    bins, cols, k = 15_500_000, 833, 18
    x = synth.synth_states_device(bins, cols, k, seed=21)
    cnt = eng.bin_counts(x, cols, k)
    for lo in range(0, bins, 1 << 21):                                 # every label counted exactly once
        c32 = cnt[lo:lo + (1 << 21)].to(torch.int32) & 0xFFFF
        assert bool((c32.sum(dim=1) == cols).all())
    del c32
    n1, n2 = eng.expected_tables(cnt, cols)
    hist = torch.zeros(k, dtype=torch.int64, device="cuda")
    for lo in range(0, bins, 1 << 18):
        hist += torch.bincount(x[lo:lo + (1 << 18), :cols].reshape(-1).to(torch.int64), minlength=k)
    assert torch.equal(n1, hist)                                      # independent histogram of the labels
    assert int(n1.sum()) == bins * cols
    assert int(n2.sum()) == bins * cols * (cols - 1)                  # closed form, SURVEY 8a
    assert torch.equal(n2, n2.T) and bool((n2 >= 0).all())
    assert torch.equal(n2.sum(dim=1), n1 * (cols - 1))
    e2 = eng.normalize(n2)
    s2 = eng.scores_s2(cnt, cols, e2)
    assert bool(torch.isfinite(s2).all())
    # spot-check 2000 bins against the oracle
    idx = torch.randperm(bins, device="cuda")[:2000]
    xs = x[idx, :cols].cpu().numpy()
    ref = orc.s2_scores(xs, k, e2.cpu().numpy(), dtype=np.float64)
    _, s2_64 = eng.scores_s2(cnt[idx].contiguous(), cols, e2, want64=True)
    np.testing.assert_allclose(s2_64.cpu().numpy(), ref, rtol=RTOL, atol=ATOL)


# ---------------------------------------------------------- stage drivers with the CUDA provider (files)
@pytest.mark.parametrize("saliency", [1, 2])
def test_stage_drivers_write_reference_files(eng, golden, tmp_path, saliency):
    """expected.main -> expectedCombination.main -> scores.main of epilogos_b200 (CUDA provider) produce the
    reference's files: int64 temp counts, float32 exp_freq payload bit-exact, scores text (spot-diff)."""
    from test_host_stages import run_single_pipeline
    g = golden("real10_chr1_k18")
    x = g["x"]
    counts, exp, npz, text = run_single_pipeline(tmp_path, x, 18, saliency, None, gz=True)
    assert counts.dtype == np.int64 and np.array_equal(counts, g["s%d_counts" % saliency])
    assert exp.tobytes() == g["s%d_exp" % saliency].tobytes()
    assert_f32_close(npz["scoreArr"], g["s%d_scores" % saliency])
    ref_lines = g["s%d_text" % saliency].tobytes().split(b"\n")
    got_lines = text.split(b"\n")
    assert len(ref_lines) == len(got_lines)
    diff = sum(a != b for a, b in zip(ref_lines, got_lines))
    assert diff <= 2, "%d of %d text lines differ" % (diff, len(ref_lines))


# ------------------------------------------------------------------------------------------------ S3
@pytest.mark.parametrize("name", ["real10_chr1_k18", "synth_s3_c12_k15", "synth_s3_c40_k18"])
def test_s3_expected_and_scores_match_reference_goldens(eng, golden, name):
    g = golden(name)
    x, k = g["x"], int(g["num_states"])
    bins, c = x.shape
    xd = dev_states(eng, x)
    tiles, plan = eng.s3_expected_tiles(xd, c, k)
    counts, exp = eng.s3_finalize(tiles, c, k, plan["mp"], bins)
    assert counts.dtype == torch.int64 and np.array_equal(counts.cpu().numpy(), g["s3_counts"])    # tensor cores, bit-exact
    assert exp.cpu().numpy().tobytes() == g["s3_exp"].tobytes()
    # the [C][C][K][K] table normalised by the generic K4 path gives the same payload
    assert eng.normalize(counts).cpu().numpy().tobytes() == g["s3_exp"].tobytes()
    terms = eng.s3_terms(exp.reshape(-1), c, k)
    ref_terms = orc.s3_pair_terms(c, g["s3_exp"], np.float64)
    np.testing.assert_allclose(eng.s3_terms_dense(terms, c, k).cpu().numpy(), ref_terms, rtol=1e-13, atol=0)
    s32, s64 = eng.scores_s3(xd, c, k, terms, want64=True)
    ref64 = orc.s3_scores_f64(x, k, g["s3_exp"])
    np.testing.assert_allclose(s64.cpu().numpy(), ref64, rtol=RTOL, atol=ATOL)
    # the reference's own float32 result carries accumulation noise (SURVEY.md 8c): agree to 2e-2 absolute
    assert np.max(np.abs(s32.cpu().numpy() - g["s3_scores"])) < 2e-2


def test_s3_scores_with_a_non_symmetric_expected_table(eng):
    """The unordered-pair S3 kernel relies on E3[i][j][a][c] == E3[j][i][c][a] (true for every table s3Calc produces) and
    checks it on the device; a foreign table without that property must take the ordered-pair kernel and still match the
    restatement.  Also covers a table with zero entries (masked terms) and a j-block that is not full (C = 13)."""
    rng = np.random.default_rng(5)
    k, c, bins = 6, 13, 700
    x = rng.integers(0, k, size=(bins, c)).astype(np.int8)
    e3 = rng.random((c, c, k, k)).astype(np.float32)
    e3 /= e3.sum()
    e3[2, 5] = 0.0                                             # masked terms
    assert not np.array_equal(e3, e3.transpose(1, 0, 3, 2))
    xd = dev_states(eng, x)
    terms = eng.s3_terms(torch.from_numpy(e3).cuda().reshape(-1), c, k)
    _, s64 = eng.scores_s3(xd, c, k, terms, want64=True)
    np.testing.assert_allclose(s64.cpu().numpy(), orc.s3_scores_f64(x, k, e3), rtol=RTOL, atol=ATOL)
    # the symmetrised table takes the unordered-pair kernel: same restatement
    es = (0.5 * (e3.astype(np.float64) + e3.transpose(1, 0, 3, 2))).astype(np.float32)
    es = np.maximum(es, es.transpose(1, 0, 3, 2))             # float32 rounding of the two halves made identical
    assert np.array_equal(es, es.transpose(1, 0, 3, 2))
    terms = eng.s3_terms(torch.from_numpy(es).cuda().reshape(-1), c, k)
    _, s64 = eng.scores_s3(xd, c, k, terms, want64=True)
    np.testing.assert_allclose(s64.cpu().numpy(), orc.s3_scores_f64(x, k, es), rtol=RTOL, atol=ATOL)


def test_s3_chunked_accumulation_and_odd_sizes(eng):
    rng = np.random.default_rng(31)
    k, c, bins = 7, 23, 1111                        # CK = 161 -> one 256 block; bins not a multiple of 128
    x = rng.integers(0, k, size=(bins, c)).astype(np.int8)
    xd = dev_states(eng, x)
    ref = orc.s3_expected_counts(x, k)
    for chunk in (None, 128, 384):
        tiles, plan = eng.s3_expected_tiles(xd, c, k, chunk_bins=chunk)
        counts, exp = eng.s3_finalize(tiles, c, k, plan["mp"], bins)
        assert np.array_equal(counts.cpu().numpy(), ref)
        assert exp.cpu().numpy().tobytes() == orc.normalize_expected(ref).tobytes()
    n3 = counts.cpu().numpy()
    assert int(n3.sum()) == bins * c * (c - 1) and np.array_equal(n3, n3.transpose(1, 0, 3, 2))
    assert not n3[np.arange(c), np.arange(c)].any()


def test_s3_benchmark_width_matches_reference_digest(eng, golden):
    """833 biosamples x 18 states (BASELINE config 3 width): 15104^2 Gram, 3540 tensor-core tiles."""
    import hashlib
    g = golden("synth_s3_c833_k18")
    x, k = g["x"], int(g["num_states"])
    bins, c = x.shape
    xd = dev_states(eng, x)
    tiles, plan = eng.s3_expected_tiles(xd, c, k)
    counts, exp = eng.s3_finalize(tiles, c, k, plan["mp"], bins)
    idx = torch.from_numpy(g["sample_idx"]).cuda()
    assert np.array_equal(counts.reshape(-1)[idx].cpu().numpy(), g["counts_sample"])
    assert np.array_equal(exp.reshape(-1)[idx].cpu().numpy(), g["exp_sample"])
    assert int(counts.sum()) == bins * c * (c - 1)
    assert hashlib.sha256(exp.cpu().numpy().tobytes()).digest() == g["exp_sha256"].tobytes()
    assert hashlib.sha256(counts.cpu().numpy().tobytes()).digest() == g["counts_sha256"].tobytes()
    terms = eng.s3_terms(exp.reshape(-1), c, k)
    s32, s64 = eng.scores_s3(xd, c, k, terms, want64=True)
    assert np.max(np.abs(s32.cpu().numpy() - g["s3_scores"])) < 2e-2
    ref64 = orc.s3_scores_f64(x, k, exp.cpu().numpy())                    # all 48 bins of the golden
    np.testing.assert_allclose(s64.cpu().numpy(), ref64, rtol=RTOL, atol=ATOL)


def test_s3_stage_drivers(eng, golden, tmp_path):
    from test_host_stages import run_single_pipeline
    g = golden("synth_s3_c12_k15")
    counts, exp, npz, text = run_single_pipeline(tmp_path, g["x"], 15, 3, None)
    assert counts.dtype == np.int64 and np.array_equal(counts, g["s3_counts"])
    assert exp.tobytes() == g["s3_exp"].tobytes()
    assert np.max(np.abs(npz["scoreArr"] - g["s3_scores"])) < 2e-2


def test_k5_tensor_core_fixed_point_table_and_scores(eng):
    """The S2 score kernel multiplies the count bytes with the base-256 digits of the 56-bit fixed-point image M of -log2 E
    on the tensor cores (kind::i8, int32 accumulators: exact).  The table it uses must be that image, F = 56 - ib fraction
    bits with -log2 E < 2^ib, and the scores must match the oracle for random, sparse and extreme count rows (all labels in
    one state, counts 0 / 1 / width - 1), for 18-, 16-, 15- and 7-state models up to the widest input of the kernel."""
    for k, width, seed in ((18, 833, 1), (15, 127, 2), (18, 1023, 3), (7, 500, 4), (16, 1000, 5), (18, 2047, 6)):
        rng = np.random.default_rng(seed)
        bins = 3000
        # count rows that sum to `width`: multinomial with random sparsity, plus extremes
        p = rng.dirichlet(np.full(k, 0.3), size=bins)
        cnt = np.stack([rng.multinomial(width, pi) for pi in p]).astype(np.int64)
        cnt[0] = 0; cnt[0, 0] = width
        cnt[1] = 0; cnt[1, k - 1] = width
        cnt[2] = 0; cnt[2, : 2] = (1, width - 1)
        e = rng.random((k, k)).astype(np.float64) ** 4 + 1e-9
        e = (e / e.sum()).astype(np.float32)
        ed = torch.from_numpy(e).cuda()
        perms = width * (width - 1)
        m, fbits = eng.scores_s2_fixed_point(ed, k, perms)
        m = m.cpu().numpy().astype(np.int64)
        assert 44 <= fbits <= 55 and m.min() >= 0 and m.max() < 2 ** 56
        want = np.rint(np.ldexp(-np.log2(e.astype(np.float64)), fbits))
        assert np.abs(m - want).max() <= 16                      # device log2 vs numpy log2: an ulp or two of a 53-bit value
        cd = torch.from_numpy(cnt.astype(np.uint16).view(np.int16)).cuda()
        ref64 = orc.s2_scores_from_counts(cnt, perms, e, dtype=np.float64)
        _, s64 = eng.scores_s2(cd, width, ed, perms=perms, want64=True)
        np.testing.assert_allclose(s64.cpu().numpy(), ref64, rtol=RTOL, atol=ATOL)


# ------------------------------------------------------------------------------------------------ paired
@pytest.mark.parametrize("k", [5, 8, 15, 18, 25])
def test_pairwise_combine_is_bitwise_numpy(eng, k):
    """delta and signed squared null distance reproduce numpy's float32 arithmetic and pairwise summation order
    (scores.py:223-232) bit for bit."""
    rng = np.random.default_rng(k)
    a, b, c, d = [(rng.standard_normal((3000, k)) * rng.choice([1e-3, 1.0, 30.0], size=(3000, 1))).astype(np.float32)
                  for _ in range(4)]
    c[:5] = d[:5]                                             # exact zeros -> sign 0
    delta, dist = eng.pairwise_combine(*[torch.from_numpy(t).cuda() for t in (a, b, c, d)])
    nd = c - d
    ref = np.sum(np.square(nd), axis=1) * np.sign(np.sum(nd, axis=1))
    assert delta.cpu().numpy().tobytes() == (a - b).tobytes()
    assert dist.cpu().numpy().tobytes() == ref.tobytes()


PAIRED_GOLDENS = ["paired_real10_k18", "paired_synth_c30_c25_k18", "paired_synth_g20_k18", "paired_synth_q0_k18",
                  "paired_synth_g40_k18"]


@pytest.mark.parametrize("name", PAIRED_GOLDENS)
def test_paired_stage_driver_replays_seeded_reference(eng, golden, tmp_path, name):
    """Supplied-permutation mode (SURVEY 8c): tables, quiescence mask, null distances and the pairwiseDelta text of a
    seeded reference run are reproduced BYTE FOR BYTE by the CUDA path, for S1 (exact value table) and for S2 (term-by-term
    float64 evaluation, which the paired driver selects in this mode)."""
    from test_host_stages import run_paired_pipeline
    g = golden(name)
    for s in (1, 2):
        if "s%d_counts" % s not in g.files:
            continue
        sub = tmp_path / ("s%d" % s)
        sub.mkdir()
        counts, exp, null, quies, text = run_paired_pipeline(sub, g["xa"], g["xb"], int(g["num_states"]), s, None,
                                                             int(g["seed"]), int(g["group_size"]),
                                                             int(g["quiescent_state"]))
        assert np.array_equal(counts, g["s%d_counts" % s]) and exp.tobytes() == g["s%d_exp" % s].tobytes()
        assert np.array_equal(quies, g["s%d_quiescence" % s])
        ref_null = g["s%d_null" % s]
        assert null.dtype == np.float32 and null.shape == ref_null.shape
        assert null.tobytes() == ref_null.tobytes(), "S%d null distances: %d of %d differ" % (
            s, int((null != ref_null).sum()), null.size)
        assert text == g["s%d_delta_text" % s].tobytes(), "S%d pairwiseDelta text differs" % s


@pytest.mark.parametrize("name", ["paired_real10_k18", "paired_synth_c30_c25_k18"])
def test_paired_s2_table_mode_is_within_one_ulp_and_rare(eng, golden, name):
    """The default (tensor-core TABLE) S2 evaluation against the exact term-by-term one on the four count arrays of the
    paired path (A, B and the replayed shuffles A', B'): float64 within 1e-9, float32 equal except 1-ulp rounding-boundary
    cases, whose rate is bounded here (measured: a few per million values)."""
    g = golden(name)
    xa, xb, k = g["xa"], g["xb"], int(g["num_states"])
    c1, c2 = xa.shape[1], xb.shape[1]
    perm = orc.reference_shuffle_indices(int(g["seed"]), xa.shape[0], c1 + c2)
    sa, sb = orc.paired_split(xa, xb, perm, -1)
    exp = torch.from_numpy(g["s2_exp"]).cuda()
    total = diff = 0
    for m, w in ((xa, c1), (xb, c2), (sa, c1), (sb, c2)):
        cnt = eng.bin_counts(dev_states(eng, np.ascontiguousarray(m)), w, k)
        t32, t64 = eng.scores_s2(cnt, w, exp, want64=True, mode=eng.EPI_SCORE_TABLE)
        d32, d64 = eng.scores_s2(cnt, w, exp, want64=True, mode=eng.EPI_SCORE_DIRECT)
        np.testing.assert_allclose(t64.cpu().numpy(), d64.cpu().numpy(), rtol=RTOL, atol=ATOL)
        assert_f32_close(t32.cpu().numpy(), d32.cpu().numpy(), max_ulp_frac=1e-4)
        total += t32.numel()
        diff += int((t32 != d32).sum())
    print("S2 TABLE vs DIRECT float32: %d of %d values differ (1 ulp)" % (diff, total))
    assert diff <= max(2, total * 1e-4)


def test_device_shuffle_is_a_uniform_split(eng):
    """Philox selection sampling: exact group sizes, never more than available, hypergeometric means, keyed by
    (seed, bin, permutation) only."""
    rng = np.random.default_rng(3)
    k, c1, c2, bins, nperm = 18, 40, 33, 600, 64
    xa = rng.integers(0, k, size=(bins, c1)).astype(np.int8)
    xb = rng.integers(0, 6, size=(bins, c2)).astype(np.int8)
    ca = eng.bin_counts(dev_states(eng, xa), c1, k)
    cb = eng.bin_counts(dev_states(eng, xb), c2, k)
    oa, ob = eng.shuffled_counts_philox(ca, cb, c1, c2, seed=99, nperm=nperm)
    oa_n, ob_n = eng.counts_to_numpy(oa).astype(np.int64), eng.counts_to_numpy(ob).astype(np.int64)
    comb = (eng.counts_to_numpy(ca).astype(np.int64) + eng.counts_to_numpy(cb).astype(np.int64))[None]
    assert (oa_n.sum(-1) == c1).all() and (ob_n.sum(-1) == c2).all()
    assert ((oa_n + ob_n) == comb).all()                       # full-size groups: every label lands somewhere
    mean = oa_n.mean(axis=0)                                    # E[a'_s] = c1 * c_s / N
    expect = c1 * comb[0] / (c1 + c2)
    assert np.abs(mean - expect).max() < 1.5                    # sd of the mean ~ 0.35 at 64 permutations
    var = oa_n.var(axis=0)                                      # Var[a'_s] = n p (1-p) (N-n)/(N-1)
    nn = c1 + c2
    pp = comb[0] / nn
    vexp = c1 * pp * (1 - pp) * (nn - c1) / (nn - 1)
    assert np.abs(var.mean(axis=0) - vexp.mean(axis=0)).max() < 0.25 * vexp.mean(axis=0).max() + 0.05
    again, _ = eng.shuffled_counts_philox(ca, cb, c1, c2, seed=99, nperm=8)
    assert torch.equal(again, oa[:8])
    other, _ = eng.shuffled_counts_philox(ca, cb, c1, c2, seed=100, nperm=8)
    assert not torch.equal(other, oa[:8])
    # -g style sub-groups: sizes respected, leftovers unassigned
    ga, gb = eng.shuffled_counts_philox(ca, cb, 20, 20, seed=5, nperm=4, width=c1 + c2)
    ga_n, gb_n = eng.counts_to_numpy(ga).astype(np.int64), eng.counts_to_numpy(gb).astype(np.int64)
    assert (ga_n.sum(-1) == 20).all() and (gb_n.sum(-1) == 20).all() and ((ga_n + gb_n) <= comb).all()


@pytest.mark.parametrize("N,K,n", [(55, 20, 30), (833, 500, 400), (833, 3, 400), (833, 830, 433), (1000, 10, 990),
                                   (15, 7, 7), (833, 417, 20), (2000, 1000, 1000)])
def test_device_hypergeometric_goodness_of_fit(eng, N, K, n):
    """Chi-square goodness of fit of the device sampler against scipy.stats.hypergeom: a two-state bin with counts
    (K, N - K) and a first group of n labels makes a'_0 ~ HG(N, K, n).  1e6 draws; cells with expectation < 10 are pooled
    into the tails.  Also with -g style sub-groups (second draw from what the first left)."""
    from scipy import stats
    bins, nperm = 1000, 1000
    ca = torch.zeros((bins, 2), dtype=torch.int16, device="cuda")
    cb = torch.zeros((bins, 2), dtype=torch.int16, device="cuda")
    ka = K // 2
    ca[:, 0] = ka; cb[:, 0] = K - ka
    na = (N - K) // 3
    ca[:, 1] = na; cb[:, 1] = N - K - na
    oa, ob = eng.shuffled_counts_philox(ca, cb, n, N - n, seed=1234 + N, nperm=nperm, width=N)
    draws = eng.counts_to_numpy(oa)[..., 0].astype(np.int64).ravel()
    lo, hi = max(0, n - (N - K)), min(n, K)
    assert draws.min() >= lo and draws.max() <= hi
    obs = np.bincount(draws - lo, minlength=hi - lo + 1).astype(np.float64)
    pmf = stats.hypergeom(N, K, n).pmf(np.arange(lo, hi + 1))
    exp_c = pmf * draws.size

    def pooled(o, e):
        keep = np.flatnonzero(e >= 10)
        a, b = keep[0], keep[-1]
        oo = np.concatenate(([o[:a + 1].sum()], o[a + 1:b], [o[b:].sum()])) if b > a else np.array([o.sum()])
        ee = np.concatenate(([e[:a + 1].sum()], e[a + 1:b], [e[b:].sum()])) if b > a else np.array([e.sum()])
        return oo, ee
    oo, ee = pooled(obs, exp_c)
    if len(oo) > 1:
        chi2 = float(((oo - ee) ** 2 / ee).sum())
        p = float(stats.chi2.sf(chi2, len(oo) - 1))
        assert p > 1e-4, "chi-square %.1f on %d cells, p = %.2e" % (chi2, len(oo), p)
    # the tails beyond float32 resolution are reachable: the smallest probability observed is consistent with 1/draws
    assert obs[pmf * draws.size < 1e-3].sum() <= 3
    # second group: b'_0 | a'_0 ~ HG(N - n, K - a'_0, m) -- check its unconditional mean and variance via a'_0 + b'_0 ~ HG(N, K, n + m)
    m = min(N - n, max(1, n // 2))
    ga, gb = eng.shuffled_counts_philox(ca, cb, n, m, seed=77 + N, nperm=200, width=N)
    tot = (eng.counts_to_numpy(ga)[..., 0].astype(np.int64) + eng.counts_to_numpy(gb)[..., 0].astype(np.int64)).ravel()
    both = stats.hypergeom(N, K, n + m)
    lo2, hi2 = max(0, n + m - (N - K)), min(n + m, K)
    obs2 = np.bincount(tot - lo2, minlength=hi2 - lo2 + 1).astype(np.float64)
    oo, ee = pooled(obs2, both.pmf(np.arange(lo2, hi2 + 1)) * tot.size)
    if len(oo) > 1:
        p = float(stats.chi2.sf(float(((oo - ee) ** 2 / ee).sum()), len(oo) - 1))
        assert p > 1e-4, "second-group chi-square p = %.2e" % p


@pytest.mark.parametrize("name,s", [("paired_synth_c30_c25_k18", 1), ("paired_synth_c30_c25_k18", 2),
                                    ("paired_real10_k18", 1), ("paired_synth_g20_k18", 1)])
def test_device_null_distances_have_the_reference_distribution(eng, golden, name, s):
    """Two-sample Kolmogorov-Smirnov test: null distances from device-drawn shuffles (64 per bin) against null distances of
    replayed reference shuffles (argsort(rand), 64 seeds per bin) on the paired goldens -- same bins, same tables."""
    from scipy import stats
    g = golden(name)
    xa, xb, k, gs = g["xa"][:300], g["xb"][:300], int(g["num_states"]), int(g["group_size"])
    c1, c2 = xa.shape[1], xb.shape[1]
    from epilogos_b200.pairwise import shuffled_widths
    wa, wb = shuffled_widths(c1, c2, gs)
    exp_np = g["s%d_exp" % s]
    exp = torch.from_numpy(exp_np).cuda()
    p1, p2 = c1 * (c1 - 1), c2 * (c2 - 1)
    ca = eng.bin_counts(dev_states(eng, xa), c1, k)
    cb = eng.bin_counts(dev_states(eng, xb), c2, k)
    nperm = 64
    oa, ob = eng.shuffled_counts_philox(ca, cb, wa, wb, seed=2024, nperm=nperm, width=c1 + c2)
    score = (lambda c, w, p: eng.scores_s1(c, max(w, 1), exp)) if s == 1 else \
        (lambda c, w, p: eng.scores_s2(c, max(w, 1), exp, perms=p))
    _, dev_null = eng.pairwise_combine(None, None, score(oa.reshape(-1, k), wa, p1), score(ob.reshape(-1, k), wb, p2))
    dev_null = dev_null.cpu().numpy()
    ref_null = []
    for seed in range(nperm):
        perm = orc.reference_shuffle_indices(1000 + seed, xa.shape[0], c1 + c2)
        r = orc.paired_scores(xa, xb, perm, k, s, exp_np, int(g["quiescent_state"]), gs)
        ref_null.append(r["null_distances"])
    ref_null = np.concatenate(ref_null)
    ks = stats.ks_2samp(dev_null, ref_null)
    print("KS statistic %.4f, p = %.3f; 1%% / 99%% quantiles device %.3f / %.3f, reference %.3f / %.3f" % (
        ks.statistic, ks.pvalue, np.quantile(dev_null, 0.01), np.quantile(dev_null, 0.99), np.quantile(ref_null, 0.01),
        np.quantile(ref_null, 0.99)))
    assert ks.pvalue > 1e-4, "KS statistic %.4f, p = %.2e" % (ks.statistic, ks.pvalue)
    assert abs(np.mean(dev_null) - np.mean(ref_null)) < 4 * np.std(ref_null) / np.sqrt(ref_null.size) * 2 + 1e-9
    for q, tol in ((0.01, 0.75), (0.05, 0.4), (0.95, 0.4), (0.99, 0.75)):      # the tails feed the p-values downstream
        assert abs(np.quantile(dev_null, q) - np.quantile(ref_null, q)) < tol * np.std(ref_null) + 1e-9


def test_paired_stage_driver_device_null(eng, golden, tmp_path):
    """Default (device-drawn) null: same delta / quiescence files, null distances with the right distribution."""
    from test_host_stages import run_paired_pipeline
    g = golden("paired_synth_c30_c25_k18")
    counts, exp, null, quies, text = run_paired_pipeline(tmp_path, g["xa"], g["xb"], 18, 1, None, 0, null_mode="device")
    assert np.array_equal(quies, g["s1_quiescence"])
    ref = g["s1_null"]
    assert null.shape == ref.shape and null.dtype == np.float32
    qs = [0.1, 0.25, 0.5, 0.75, 0.9]
    assert np.abs(np.quantile(null, qs) - np.quantile(ref, qs)).max() < 0.35 * np.std(ref)


def test_paired_real_reductions_with_text_round_trip(eng):
    """f2: distance + max-difference state of the real deltas exactly as the reference's paired ROI stage sees them
    after re-parsing the 5-decimal text (roiAndVisualPairwise.py:339-354), without writing or reading any text."""
    rng = np.random.default_rng(8)
    k = 18
    d = (rng.standard_normal((20000, k)) * rng.choice([1e-4, 1e-2, 1.0, 50.0], size=(20000, 1))).astype(np.float32)
    d[:50] = np.float32(1.0 / 64)                      # exact decimal ties: 0.015625 -> "0.01562"
    d[50:100] = np.float32(3.0 / 64) * np.float32(-1)  # -0.046875 -> "-0.04688"
    d[100:120] = 0
    d[120:140, 3] = np.float32(-1e-7)                   # prints "-0.00000"
    ref_dist, ref_md = orc.paired_real_reductions(d)
    dist, md = eng.pairwise_real_reduce(torch.from_numpy(d).cuda(), text_round_trip=True)
    assert dist.cpu().numpy().tobytes() == ref_dist.tobytes()
    assert np.array_equal(md.cpu().numpy(), ref_md)
    ref_dist, ref_md = orc.paired_real_reductions(d, round_trip=False)
    dist, md = eng.pairwise_real_reduce(torch.from_numpy(d).cuda(), text_round_trip=False)
    assert dist.cpu().numpy().tobytes() == ref_dist.tobytes() and np.array_equal(md.cpu().numpy(), ref_md)


def test_s3_chr1_shape_properties(eng):
    """BASELINE configs[2] at full size (1.25 M bins x 833 biosamples x 18 states): closed-form total, empty diagonal
    blocks and one pair of the tensor-core Gram table; scores of a sample against the float64 oracle.  (The table is
    symmetric by construction of epi_s3_finalize; tests/test_s3_gpu.py compares whole tables in steady state.)"""
    from epilogos_b200 import synth
    bins, cols, k = 1_250_000, 833, 18
    x = synth.synth_states_device(bins, cols, k, seed=22)
    tiles, plan = eng.s3_expected_tiles(x, cols, k)
    counts, exp = eng.s3_finalize(tiles, cols, k, plan["mp"], bins)
    assert int(counts.sum()) == bins * cols * (cols - 1)                         # SURVEY 8a closed form
    idx = torch.arange(cols, device="cuda")
    assert not bool(counts[idx, idx].any())                                      # i == j blocks stay empty
    # pair (0, 1): against a direct 2-D histogram of the two label columns
    pair = torch.bincount(x[:, 0].long() * k + x[:, 1].long(), minlength=k * k).reshape(k, k)
    assert torch.equal(counts[0, 1], pair)
    assert abs(float(exp.double().sum()) - 1.0) < 1e-6
    terms = eng.s3_terms(exp.reshape(-1), cols, k)
    # 256 bins drawn at random from the whole chromosome (plus the first and the last bin) against the float64 restatement
    pick = np.sort(np.random.default_rng(77).choice(bins, size=254, replace=False))
    pick = np.concatenate(([0], pick, [bins - 1]))
    sub = x[torch.from_numpy(pick).cuda()].contiguous()
    s32, s64 = eng.scores_s3(sub, cols, k, terms, want64=True)
    exp_np = exp.cpu().numpy()
    t64 = orc.s3_pair_terms(cols, exp_np, np.float64)
    ref = orc.s3_scores_f64(sub[:, :cols].cpu().numpy(), k, exp_np, terms=t64)
    np.testing.assert_allclose(s64.cpu().numpy(), ref, rtol=RTOL, atol=ATOL)
    assert np.max(np.abs(s32.cpu().numpy().astype(np.float64) - ref)) < 1e-5
    assert bool(torch.isfinite(s32).all())


def test_two_gpu_stage_drivers_match_goldens(eng):
    """Rows sharded over 2 ranks (NCCL): same files as the single-process reference goldens (tools/mgpu_check.py)."""
    import subprocess
    import sys
    from pathlib import Path
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import os
    root = Path(__file__).resolve().parent.parent
    # rows of every file over the ranks, read by every rank itself (the path measured in round 2) and dealt by one reader
    # rank per file (opt-in over NCCL until this test has passed on hardware: its NCCL branch was written without a GPU)
    for port, mode in ((29577, "redundant"), (29578, "deal")):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", str(port), str(root / "tools" / "mgpu_check.py")],
                           capture_output=True, text=True, timeout=600, env=dict(os.environ, EPILOGOS_B200_READ=mode))
        assert "MGPU ALL OK" in r.stdout, "EPILOGOS_B200_READ=%s\n" % mode + r.stdout[-3000:] + r.stderr[-3000:]
