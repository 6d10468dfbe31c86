"""S1 and S2 score kernels (K5) against independent float64 references on every bin, every tile and every launch.

The references are plain torch float64 from the count rows: S1 o = c / width, S2 o_st = (c_s c_t - [s=t] c_s) / P,
term = o log2(o / E), 0 where o = 0 or E = 0 (klScoreND's masking), S2 terms added over s in order.  Neither uses the
library's tables, its TABLE algebra or its kernels; both are pinned to the numpy oracle in a CPU-only test.

Every case calls the library three times through the C ABI, into views of buffers padded with sentinel rows: with both
outputs (the WANT64 kernel instances), float32 only (the instances production runs) and float64 only.  s2_route,
tc_schedule and k5_schedule restate the launch choices of csrc/scores.cu and csrc/tc_tables.cu, so the CPU-only tests
below show which kernel instance and which schedule each case reaches, and a failure names the tile, CTA and warpgroup
(or warp) that owns the bin.  Count rows are drawn on the device from a seeded torch.Generator.
"""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import epilogos_oracle as orc            # noqa: E402  (checker only)
from test_limits_gpu import s1_launch                 # noqa: E402

RTOL, ATOL = 1e-9, 1e-12
TABLE, DIRECT = 0, 1          # EPI_SCORE_TABLE, EPI_SCORE_DIRECT
PAD = 64                      # sentinel rows before and after every output
SENT32 = 0x7fa0dead           # NaN bit patterns no kernel writes
SENT64 = 0x7ff4deadbeef0bad
B200_SMS = 148                # SM count the CPU-only coverage tests assume


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import build, engine
    build.build()
    engine.device_info()
    return engine


@pytest.fixture(scope="module")
def sms(eng):
    return torch.cuda.get_device_properties(0).multi_processor_count


def u16(cnt):
    """int16 tensor holding uint16 counts -> int64 tensor of the counts."""
    return cnt.to(torch.int64) & 0xffff


# ------------------------------------------------------------------------------------------------ references
def s1_reference(cnt, width, exp1, chunk=1 << 22):
    """float64 [bins, K]: o log2(o / E[s]) with o = c / width; 0 where o = 0 or E = 0."""
    e = exp1.to(torch.float64).reshape(1, -1)
    out = torch.empty(cnt.shape, dtype=torch.float64, device=cnt.device)
    for lo in range(0, cnt.shape[0], chunk):
        o = u16(cnt[lo:lo + chunk]).to(torch.float64) / width
        out[lo:lo + o.shape[0]] = torch.where((o == 0) | (e == 0), 0.0, o * torch.log2(o / e))
    return out


def s2_reference(cnt, perms, exp2, chunk_elems=1 << 24):
    """float64 [bins, K]: sum over s = 0..K-1, in order, of o_st log2(o_st / E_st) with o_st = (c_s c_t - [s=t] c_s) / P;
    a term is 0 where o = 0 or E = 0.  The products are exact in float64 (below 2^32)."""
    k = cnt.shape[1]
    e = exp2.to(torch.float64).reshape(1, k, k)
    idx = torch.arange(k, device=cnt.device)
    out = torch.empty(cnt.shape, dtype=torch.float64, device=cnt.device)
    chunk = max(1, chunk_elems // (k * k))
    for lo in range(0, cnt.shape[0], chunk):
        c = u16(cnt[lo:lo + chunk]).to(torch.float64)
        prod = c[:, :, None] * c[:, None, :]
        prod[:, idx, idx] -= c
        o = prod / perms
        term = torch.where((o == 0) | (e == 0), 0.0, o * torch.log2(o / e))
        acc = torch.zeros_like(c)
        for s in range(k):
            acc += term[:, s, :]
        out[lo:lo + c.shape[0]] = acc
    return out


# ------------------------------------------------------------------------------------------------ launch restatements
def s2_kt(k):
    return 16 if k <= 16 else 18 if k <= 18 else 32


def s2_tc_instance(k):
    """<KT, KR, NWG> of k5_s2_tc_kernel that scores_s2_tc (csrc/tc_tables.cu) picks."""
    if k == 18:
        return (18, 18, 3)
    if k == 15:
        return (16, 15, 4)
    return (16, 0, 4) if k <= 16 else (18, 0, 3) if k <= 18 else (32, 0, 2)


def s2_route(k, width, mode, table_has_zero):
    """The kernel that writes the S2 scores (epi_scores_s2 / dispatch_s2, csrc/scores.cu): the tensor-core instance for
    TABLE at width <= 2047 (T5_MAX_WIDTH), or the DIRECT k5_s2_kernel<KT> queued behind it and gated on the table's zero
    flag; the DFMA TABLE form of k5_s2_kernel<KT> above 2047, which turns itself into DIRECT on that flag; DIRECT."""
    kt = s2_kt(k)
    if mode == TABLE and width <= 2047:
        return ("gated",) + s2_tc_instance(k) if table_has_zero else ("tc",) + s2_tc_instance(k)
    if mode == TABLE and not table_has_zero:
        return ("dfma", kt)
    return ("direct", kt)


def tc_schedule(bins, nwg, sms):
    """The schedule of k5_s2_tc_kernel: 128-bin tiles, grid = min(tiles, SMs) CTAs, warpgroup g of CTA b takes the tiles
    b + g grid + u NWG grid; the producer bulk-loads only full tiles, the partial last tile is read with plain loads."""
    tiles = -(-bins // 128)
    grid = max(1, min(tiles, sms))
    per = [max(0, -(-(tiles - (b + g * grid)) // (nwg * grid))) for b in range(grid) for g in range(nwg)]
    partial = None
    if bins % 128:
        t = tiles - 1
        partial = (t % grid, (t // grid) % nwg)
    return dict(tiles=tiles, grid=grid, min_tiles=min(per), max_tiles=max(per), partial=partial)


def tc_owner(b, bins, nwg, sms):
    grid = max(1, min(-(-bins // 128), sms))
    t = b // 128
    return "tile %d, CTA %d, warpgroup %d, warp %d" % (t, t % grid, (t // grid) % nwg, (b % 128) // 32)


def k5_schedule(bins, threads, per_sm, sms):
    """The per-warp streams of k5_s2_kernel and k5_s1_kernel (WarpCountStream): 32-bin groups, grid =
    min(ceil(bins / threads), per_sm SMs) CTAs, warp w of CTA b takes the groups b W + w + i grid W (W = threads / 32);
    full groups arrive by bulk copies into two slabs, the partial last group by plain loads."""
    groups = -(-bins // 32)
    grid = max(1, min(-(-bins // threads), per_sm * sms))
    nw = grid * (threads // 32)
    partial = None
    if bins % 32:
        g = groups - 1
        partial = ((g % nw) // (threads // 32), g % (threads // 32))
    return dict(groups=groups, grid=grid, min_groups=groups // nw, max_groups=-(-groups // nw), partial=partial)


def k5_owner(b, bins, threads, per_sm, sms):
    grid = max(1, min(-(-bins // threads), per_sm * sms))
    w, g = threads // 32, b // 32
    return "group %d, CTA %d, warp %d, pass %d" % (g, (g % (grid * w)) // w, g % w, g // (grid * w))


S2_STREAM = (256, 3)          # k5_s2_kernel: K5_THREADS, persistent_grid(ntiles, 3)


def s1_stream(name):
    """(threads, CTAs per SM) of a launch of launch_s1 (as s1_launch names it); None for the per-element DIRECT kernel."""
    if name == "direct":
        return None
    if name == "smem, 1024 threads":
        return (1024, 1)
    if name == "global table":
        return (256, 4)
    return (256, int(name.split(" x ")[1].split()[0]))


def owner(route, b, bins, k, sms):
    """Who writes bin b: tile / CTA / warpgroup / warp of the restated schedule."""
    if route[0] == "tc":
        return tc_owner(b, bins, route[3], sms)
    if route[0] in ("gated", "dfma", "direct"):
        return k5_owner(b, bins, *S2_STREAM, sms)
    if route[0] == "s1":
        st = s1_stream(route[2])
        if st is not None:
            return k5_owner(b, bins, *st, sms)
    grid = max(1, min(-(-bins * k // 256), 16 * sms))
    return "elements %d..%d, CTA %d" % (b * k, b * k + k - 1, (b * k // 256) % grid)


def per_sms(a, b):
    """bins = a x SMs + b."""
    return (a, b)


def tc_steady(nwg, last):
    """At least 5 tiles per warpgroup, and a partial last tile owned by warpgroup 0 of CTA 5 or by warpgroup NWG - 1 of
    CTA 7."""
    q, r, extra = (6 * nwg - 1, 7, 33) if last else (5 * nwg, 5, 77)
    return per_sms(128 * q, 128 * r + extra)


def stream_steady(threads, per_sm):
    """At least 5 groups per warp of a per-warp-stream launch, and a partial last group on CTA 5."""
    return per_sms(5 * threads * per_sm, 32 * (5 * threads // 32 + 3) + 19)


def case_bins(spec, sms):
    return spec[0] * sms + spec[1]


# ------------------------------------------------------------------------------------------------ cases
# S2: (K, width, perms or None for width (width - 1), bins = (a, b) for a SMs + b, table, rows, mode).  The perms of a
# paired run under -g: null rows of `width` biosamples normalised with c1 (c1 - 1) for the group's real size c1.
S2_CASES = [
    # every tensor-core instance in steady state, the partial tile on warpgroup 0 and on warpgroup NWG - 1
    (18, 833, None, tc_steady(3, False), "data", "mixed", TABLE),
    (18, 2047, None, tc_steady(3, True), "near128", "one", TABLE),
    (15, 127, None, tc_steady(4, False), "data", "mixed", TABLE),
    (15, 255, None, tc_steady(4, True), "subnormal", "mixed", TABLE),
    (16, 256, None, tc_steady(4, False), "dir4", "mixed", TABLE),
    (7, 10, None, tc_steady(4, True), "pow2", "mixed", TABLE),
    (17, 2047, None, tc_steady(3, False), "near128", "one", TABLE),
    (17, 833, None, tc_steady(3, True), "data", "mixed", TABLE),
    (25, 127, None, tc_steady(2, False), "dir4", "mixed", TABLE),
    (32, 2047, None, tc_steady(2, True), "near128", "one", TABLE),
    # one bin, no full tile, exact multiples of 128, fewer tiles than SMs
    (18, 10, None, per_sms(0, 1), "dir4", "mixed", TABLE),
    (1, 2, None, per_sms(0, 77), "dir4", "mixed", TABLE),
    (2, 2, None, per_sms(0, 127), "data", "mixed", TABLE),
    (16, 256, None, per_sms(0, 128), "subnormal", "mixed", TABLE),
    (19, 255, None, per_sms(0, 128 * 40), "subnormal", "mixed", TABLE),
    (31, 833, None, per_sms(0, 128 * 100 + 5), "pow2", "mixed", TABLE),
    (2, 127, None, per_sms(128, 1), "dir4", "mixed", TABLE),
    (1, 2047, None, per_sms(0, 3001), "near128", "one", TABLE),
    # perms of -g null rows, c1 above and below the width
    (18, 10, 12 * 11, per_sms(0, 5001), "data", "mixed", TABLE),
    (18, 10, 8 * 7, per_sms(0, 5001), "dir4", "mixed", TABLE),
    (15, 127, 130 * 129, per_sms(0, 3001), "data", "mixed", TABLE),
    (15, 127, 100 * 99, per_sms(0, 3001), "pow2", "mixed", TABLE),
    (7, 2100, 2200 * 2199, per_sms(0, 4001), "data", "mixed", TABLE),
    (25, 2048, 2000 * 1999, per_sms(0, 4001), "dir4", "mixed", TABLE),
    # tables with zero entries: the DIRECT kernel gated behind every tensor-core instance, and behind the DFMA form
    (18, 833, None, stream_steady(*S2_STREAM), "zero", "mixed", TABLE),
    (15, 127, None, per_sms(0, 3001), "zero", "mixed", TABLE),
    (7, 256, None, per_sms(0, 2001), "zero", "mixed", TABLE),
    (17, 10, None, per_sms(0, 1001), "zero", "mixed", TABLE),
    (25, 2047, None, per_sms(0, 2001), "zero", "mixed", TABLE),
    (25, 2100, None, per_sms(0, 2001), "zero", "mixed", TABLE),
    # the DFMA TABLE form of every KT, in steady state
    (7, 2048, None, stream_steady(*S2_STREAM), "dir4", "mixed", TABLE),
    (18, 2100, None, stream_steady(*S2_STREAM), "data", "mixed", TABLE),
    (32, 2100, None, stream_steady(*S2_STREAM), "pow2", "mixed", TABLE),
    (17, 2048, None, per_sms(0, 3001), "subnormal", "mixed", TABLE),
    # DIRECT of every KT
    (16, 833, None, stream_steady(*S2_STREAM), "data", "mixed", DIRECT),
    (18, 10, None, per_sms(0, 999), "dir4", "mixed", DIRECT),
    (32, 127, None, per_sms(0, 3001), "data", "mixed", DIRECT),
    (15, 255, 250 * 249, per_sms(0, 2001), "subnormal", "mixed", DIRECT),
]

# S1: (K, width, bins, table)
S1_CASES = [
    (18, 833, stream_steady(1024, 1), "data"),         # smem table, 1024 threads
    (18, 10, stream_steady(256, 4), "dir4"),           # 256 threads x 4
    (32, 10, stream_steady(256, 3), "subnormal"),      # x 3
    (25, 255, stream_steady(256, 2), "data"),          # x 2
    (18, 1200, stream_steady(256, 1), "zero"),         # x 1
    (32, 2047, stream_steady(256, 4), "dir4"),         # global table
    (15, 4096, per_sms(0, 50001), "data"),             # direct
    (1, 2, per_sms(0, 1), "dir4"),
    (2, 127, per_sms(0, 77), "data"),
    (7, 2100, per_sms(0, 3001), "subnormal"),
    (31, 256, per_sms(0, 128 * 40), "zero"),
    (16, 2048, per_sms(0, 5003), "data"),
    (17, 1332, per_sms(0, 1000), "dir4"),
    (19, 833, per_sms(0, 999), "zero"),
    (25, 5000, per_sms(0, 2001), "dir4"),
]

TABLES_WITH_ZERO = {"zero"}


def s1_route(k, width):
    return ("s1", width, s1_launch(k, width))


def s2_case_id(c):
    k, width, perms, bins, table, rows, mode = c
    return "k%d-w%d-%s-%s%s%s" % (k, width, "%dx+%d" % bins if bins[0] else str(bins[1]), table,
                                  "" if perms is None else "-p%d" % perms, "-direct" if mode == DIRECT else "")


# ------------------------------------------------------------------------------------------------ inputs
def count_rows(bins, k, width, seed, rows="mixed", device="cuda", chunk=1 << 22):
    """uint16 count rows (in int16) [bins, K] that sum to `width`: skewed random shares (half the rows drawn with every
    state likely present, half with a few dominant states), or every row in one random state."""
    g = torch.Generator(device=device).manual_seed(seed)
    out = torch.empty((bins, k), dtype=torch.int16, device=device)
    for lo in range(0, bins, chunk):
        n = min(chunk, bins - lo)
        pick = torch.randint(0, k, (n,), generator=g, device=device)
        if rows == "one":
            c = torch.zeros((n, k), dtype=torch.int64, device=device)
            c[torch.arange(n, device=device), pick] = width
        else:
            expo = torch.where(torch.rand((n, 1), generator=g, device=device) < 0.5, 1.0, 4.0).to(torch.float64)
            w = torch.rand((n, k), generator=g, device=device, dtype=torch.float64) ** expo
            c = torch.floor(w / w.sum(dim=1, keepdim=True).clamp_min(1e-300) * width).to(torch.int64)
            c[torch.arange(n, device=device), pick] += width - c.sum(dim=1)
        out[lo:lo + n] = c.to(torch.int16)
        del c
    return out


def extreme_rows(k, width):
    """Every state alone (c = width); 1 and width - 1; every state present; with width >= 256, counts above 255 in both
    bytes of the A operand."""
    rows = []
    for s in range(k):
        r = [0] * k
        r[s] = width
        rows.append(r)
        if k > 1:
            r = [0] * k
            r[s], r[(s + 1) % k] = 1, width - 1
            rows.append(r)
            if width >= 512:
                r = [0] * k
                r[s], r[(s + 1) % k] = 256 + s, width - 256 - s
                rows.append(r)
                r = [0] * k
                r[s], r[(s + 3) % k] = 255, width - 255
                rows.append(r)
    if width >= k:
        r = [width // k] * k
        r[k - 1] += width - sum(r)
        rows.append(r)
        r = [1] * k
        r[0] += width - k
        rows.append(r)
    out = np.array(rows, dtype=np.int64)
    assert (out.sum(axis=1) == width).all() and out.min() >= 0
    return out


def plant(cnt, rows):
    """The extreme rows at the start of the first tile, across the tile boundary in the middle and at the end (in the
    partial last tile)."""
    bins, n = cnt.shape[0], rows.shape[0]
    r = torch.from_numpy(rows.astype(np.int16)).to(cnt.device)
    tiles = -(-bins // 128)
    for start in (0, max(0, 128 * (tiles // 2) - n // 2), max(0, bins - n)):
        m = min(n, bins - start)
        cnt[start:start + m] = r[:m]
    return cnt


def make_counts(bins, k, width, seed, rows="mixed", device="cuda"):
    return plant(count_rows(bins, k, width, seed, rows, device), extreme_rows(k, width))


def expected_table(kind, cnt, k, s2, seed):
    """float32 expected table ([K, K] for S2, [K] for S1) on the counts' device."""
    rng = np.random.default_rng(seed)
    n = k * k if s2 else k
    if kind == "data":
        c = u16(cnt).to(torch.float64)
        if s2:
            n2 = c.T @ c - torch.diag(c.sum(dim=0))          # exact: every partial sum stays below 2^53
            return (n2 / n2.sum()).to(torch.float32).reshape(k, k).contiguous()
        n1 = c.sum(dim=0)
        return (n1 / n1.sum()).to(torch.float32)
    if kind == "near128":
        # all entries just above 2^-128 (float32 subnormals): -log2 E just below 128, M just below 2^56
        e = (2.0 ** -128 + np.arange(1, n + 1) * 2.0 ** -149).astype(np.float32)
    else:
        e = rng.dirichlet(np.ones(n))
        if kind == "dir4":
            e = e ** 4
            e /= e.sum()
            e = np.maximum(e, 2.0 ** -100)
        e = e.astype(np.float32)
        if kind == "subnormal":
            e[n // 2] = np.float32(2.0 ** -149)                 # the smallest float32 subnormal: -log2 E = 149, F = 48
        elif kind == "pow2":
            e = np.maximum(e, np.float32(2.0 ** -31))
            e[n - 1] = np.float32(2.0 ** -32)                   # the largest -log2 E is exactly 32
        elif kind == "zero":
            e[0] = 0.0
            e[n - 1] = 0.0
            if n > 4:
                e[n // 2] = 0.0
    t = torch.from_numpy(e).to(cnt.device)
    return t.reshape(k, k).contiguous() if s2 else t


def fraction_bits(e):
    """F of k5tc_prepare_kernel: 56 - ib, with ib the least integer >= 1 (at most 12) such that max -log2 E < 2^ib."""
    e = np.asarray(e, dtype=np.float64)
    mx = max(0.0, float(np.max(-np.log2(e[e > 0])))) if (e > 0).any() else 0.0
    ib = 1
    while ib < 12 and 2.0 ** ib <= mx:
        ib += 1
    return 56 - ib


# ------------------------------------------------------------------------------------------------ calls and checks
def _ptr(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def call_scores(eng, cnt, width, e, mode, perms=None, want32=True, want64=False, route=None, sms=None):
    """One call of epi_scores_s2 (perms given) or epi_scores_s1 into views of sentinel-filled buffers with PAD rows on
    either side; the padding must come back untouched.  Returns (out32 or None, out64 or None)."""
    from epilogos_b200 import _lib
    bins, k = cnt.shape
    outs = []
    for want, dt, it, sent in ((want32, torch.float32, torch.int32, SENT32), (want64, torch.float64, torch.int64, SENT64)):
        if not want:
            outs.append((None, None, None))
            continue
        buf = torch.full(((bins + 2 * PAD) * k,), sent, dtype=it, device=cnt.device)
        outs.append((buf, buf.view(dt)[PAD * k:(PAD + bins) * k].view(bins, k), sent))
    (b32, o32, _), (b64, o64, _) = outs
    if perms is None:
        _lib.call("epi_scores_s1", _ptr(cnt), bins, k, int(width), _ptr(e), _ptr(o32), _ptr(o64), int(mode), eng._stream())
    else:
        _lib.call("epi_scores_s2", _ptr(cnt), bins, k, int(width), int(perms), _ptr(e), _ptr(o32), _ptr(o64), int(mode),
                  eng._stream())
    for buf, _, sent in outs:
        if buf is None:
            continue
        pad = torch.cat([buf[:PAD * k], buf[(PAD + bins) * k:]])
        bad = (pad != sent).nonzero().flatten()
        if len(bad):
            i = int(bad[0])
            where = ("row %d before bin 0" % (i // k - PAD) if i < PAD * k else
                     "bin %d past the last bin %d (%s)" % (bins + (i - PAD * k) // k, bins - 1,
                                                           owner(route, bins + (i - PAD * k) // k, bins, k, sms)))
            raise AssertionError("%s: %d padding elements overwritten, the first at %s, state %d"
                                 % (route, len(bad), where, i % k))
    return o32, o64


def _describe(bad, got, want, route, bins, k, sms, what):
    idx = bad.nonzero()
    rows = idx[:, 0].unique()
    pos = []
    for b, s in idx[:8].tolist():
        pos.append("bin %d state %d (%s): %r, want %r" % (b, s, owner(route, b, bins, k, sms), float(got[b, s]),
                                                           float(want[b, s])))
    return "%s %s: %d of %d values differ in %d bins: %s" % (route, what, idx.shape[0], bad.numel(), rows.numel(),
                                                              "; ".join(pos))


def assert_f64_close(got, ref, route, sms):
    bad = ~torch.isclose(got, ref, rtol=RTOL, atol=ATOL)
    if bool(bad.any()):
        raise AssertionError(_describe(bad, got, ref, route, got.shape[0], got.shape[1], sms, "float64 output"))


def assert_bits_equal(got, want, route, sms, what):
    it = torch.int32 if got.dtype == torch.float32 else torch.int64
    bad = got.view(it) != want.view(it)
    if bool(bad.any()):
        raise AssertionError(_describe(bad, got, want, route, got.shape[0], got.shape[1], sms, what))


def assert_f32_rounds_reference(got32, ref, route, sms, max_ulp_frac=2e-3):
    """float32 output against the float32 rounding of the reference: equal but for rare rounding-boundary cases at most
    1 ulp apart; zeros carry the reference's sign (as assert_f32_close in test_gpu_parity)."""
    r32 = ref.to(torch.float32)
    bins, k = got32.shape
    zero = r32 == 0
    bad = zero & (torch.signbit(got32) != torch.signbit(r32))
    if bool(bad.any()):
        raise AssertionError(_describe(bad, got32, r32, route, bins, k, sms, "float32 zero sign"))
    neq = got32.view(torch.int32) != r32.view(torch.int32)
    if not bool(neq.any()):
        return
    m = torch.maximum(got32.abs(), r32.abs())
    ulp = (torch.nextafter(m, torch.full_like(m, float("inf"))) - m).to(torch.float64)
    far = neq & ~((got32.to(torch.float64) - r32.to(torch.float64)).abs() <= ulp * 1.0000001)
    if bool(far.any()):
        raise AssertionError(_describe(far, got32, r32, route, bins, k, sms, "float32 output more than 1 ulp off"))
    frac = float(neq.float().mean())
    assert frac <= max_ulp_frac, "%s: too many 1-ulp differences from the reference: %g" % (route, frac)


def check_all_outputs(eng, cnt, width, e, mode, perms, ref, route, sms):
    """The three calls of one case and every assertion on them; returns the float64 output."""
    w32, w64 = call_scores(eng, cnt, width, e, mode, perms, want32=True, want64=True, route=route, sms=sms)
    assert_f64_close(w64, ref, route, sms)
    r32 = w64.to(torch.float32)
    assert_bits_equal(w32, r32, route, sms, "float32 output of the float64 call vs the rounding of its float64 output")
    s32, _ = call_scores(eng, cnt, width, e, mode, perms, want32=True, route=route, sms=sms)
    assert_bits_equal(s32, r32, route, sms, "float32-only output vs the rounding of the float64 output")
    assert_f32_rounds_reference(s32, ref, route, sms)
    _, o64 = call_scores(eng, cnt, width, e, mode, perms, want32=False, want64=True, route=route, sms=sms)
    assert_bits_equal(o64, w64, route, sms, "float64-only output vs the float64 output")
    return s32, w64


# ------------------------------------------------------------------------------------------------ CPU-only tests
PIN_CASES = [(18, 10, None, "data"), (15, 127, 100 * 99, "dir4"), (15, 127, 130 * 129, "subnormal"),
             (32, 2047, None, "near128"), (7, 2100, 2200 * 2199, "zero"), (1, 2, None, "dir4"), (2, 256, None, "pow2"),
             (25, 833, None, "zero")]


@pytest.mark.parametrize("k,width,perms,table", PIN_CASES)
def test_references_match_the_oracle(k, width, perms, table):
    """Both references on the CPU against orc.s1_scores_from_counts / orc.s2_scores_from_counts, on a few thousand rows
    with every extreme row, to 1e-13 relative: only the log2 implementations differ."""
    cnt = make_counts(3000, k, width, seed=k * 1000 + width, device="cpu")
    c = u16(cnt).numpy()
    assert (c.sum(axis=1) == width).all()
    assert (c == width).any(axis=1).sum() >= k and (k == 1 or (c.max(axis=1) < width).any())
    p = width * (width - 1) if perms is None else perms
    e2 = expected_table(table, cnt, k, True, seed=k)
    e1 = expected_table(table, cnt, k, False, seed=k)
    want2 = orc.s2_scores_from_counts(c, p, e2.numpy(), np.float64)
    np.testing.assert_allclose(s2_reference(cnt, p, e2, chunk_elems=1 << 16).numpy(), want2, rtol=1e-13, atol=0)
    want1 = orc.s1_scores_from_counts(c, width, e1.numpy(), np.float64)
    np.testing.assert_allclose(s1_reference(cnt, width, e1).numpy(), want1, rtol=1e-13, atol=0)


def test_s2_route_table():
    assert s2_route(18, 2047, TABLE, False) == ("tc", 18, 18, 3)
    assert s2_route(15, 10, TABLE, False) == ("tc", 16, 15, 4)
    assert s2_route(16, 10, TABLE, False) == ("tc", 16, 0, 4)
    assert s2_route(17, 10, TABLE, False) == ("tc", 18, 0, 3)
    assert s2_route(19, 10, TABLE, False) == ("tc", 32, 0, 2)
    assert s2_route(17, 10, TABLE, True) == ("gated", 18, 0, 3)
    assert s2_route(18, 2048, TABLE, False) == ("dfma", 18)
    assert s2_route(18, 2048, TABLE, True) == ("direct", 18)
    assert s2_route(1, 10, DIRECT, False) == ("direct", 16)
    assert {s2_tc_instance(k) for k in range(1, 33)} == {(18, 18, 3), (16, 15, 4), (16, 0, 4), (18, 0, 3), (32, 0, 2)}


def test_schedules_on_known_shapes():
    s = tc_schedule(1, 4, 148)
    assert (s["tiles"], s["grid"], s["min_tiles"], s["max_tiles"], s["partial"]) == (1, 1, 0, 1, (0, 0))
    s = tc_schedule(128 * 148 * 3, 3, 148)
    assert (s["grid"], s["min_tiles"], s["max_tiles"], s["partial"]) == (148, 1, 1, None)
    s = tc_schedule(128 * 300 + 1, 2, 148)                 # tile 300 = CTA 4, second pass of warpgroup 0
    assert (s["tiles"], s["min_tiles"], s["max_tiles"], s["partial"]) == (301, 1, 2, (4, 0))
    assert tc_owner(128 * 300, 128 * 300 + 1, 2, 148) == "tile 300, CTA 4, warpgroup 0, warp 0"
    s = k5_schedule(32 * 100 + 5, 256, 3, 148)             # 101 groups, 13 CTAs of 8 warps
    assert (s["grid"], s["min_groups"], s["max_groups"], s["partial"]) == (13, 0, 1, (12, 4))
    assert k5_owner(32 * 100, 32 * 100 + 5, 256, 3, 148) == "group 100, CTA 12, warp 4, pass 0"


def s2_calls(case):
    """(kernel instance, WANT64) of every launch a case's three calls make that writes scores."""
    k, width, perms, bins, table, rows, mode = case
    route = s2_route(k, width, mode, table in TABLES_WITH_ZERO)
    if route[0] == "tc":
        return {(route, True), (route, False)}
    return {(route, None)}


def test_s2_cases_reach_every_kernel_instance():
    """All 10 tensor-core instances (5 <KT, KR, NWG> x WANT64), the DFMA and DIRECT forms of k5_s2_kernel<16/18/32>, and
    the DIRECT kernel gated behind every tensor-core instance."""
    reached = set().union(*(s2_calls(c) for c in S2_CASES))
    tc = [("tc",) + i for i in ((18, 18, 3), (16, 15, 4), (16, 0, 4), (18, 0, 3), (32, 0, 2))]
    want = {(r, w) for r in tc for w in (True, False)}
    want |= {(("gated",) + r[1:], None) for r in tc}
    want |= {((f, kt), None) for f in ("dfma", "direct") for kt in (16, 18, 32)}
    assert reached == want
    assert {c[0] for c in S2_CASES} >= {1, 2, 7, 15, 16, 17, 18, 19, 25, 31, 32}
    assert {c[1] for c in S2_CASES} >= {2, 10, 127, 255, 256, 833, 2047, 2048, 2100}
    assert {c[4] for c in S2_CASES} == {"data", "dir4", "subnormal", "pow2", "near128", "zero"}


def test_s2_cases_reach_steady_state_and_the_tile_edges():
    """For every tensor-core instance a case where every warpgroup of every CTA takes >= 5 tiles (both count slabs wrap
    their phases twice), with the partial tile on warpgroup 0 and on warpgroup NWG - 1 of a CTA other than 0; >= 5 groups
    per warp for every k5_s2_kernel<KT>; one bin, no full tile, exact multiples of 128, fewer tiles than SMs."""
    sms = B200_SMS
    steady, owners, edges, streams = set(), set(), set(), set()
    for c in S2_CASES:
        k, width, perms, bins, table, rows, mode = c
        route = s2_route(k, width, mode, table in TABLES_WITH_ZERO)
        b = case_bins(bins, sms)
        if route[0] == "tc":
            s = tc_schedule(b, route[3], sms)
            if s["min_tiles"] >= 5:
                steady.add(route)
            if s["partial"] and s["partial"][0] != 0:
                owners.add((route, s["partial"][1] == 0, s["partial"][1] == route[3] - 1))
            edges |= {e for e, hit in (("one bin", b == 1), ("no full tile", b < 128), ("multiple of 128", b % 128 == 0),
                                       ("fewer tiles than SMs", 1 < s["tiles"] < sms)) if hit}
        else:
            s = k5_schedule(b, *S2_STREAM, sms)
            if s["min_groups"] >= 5 and s["partial"] and s["partial"][0] != 0:
                streams.add(route[1])
    tc = {("tc",) + i for i in ((18, 18, 3), (16, 15, 4), (16, 0, 4), (18, 0, 3), (32, 0, 2))}
    assert steady == tc
    assert {r for r, first, _ in owners if first} == tc and {r for r, _, last in owners if last} == tc
    assert edges == {"one bin", "no full tile", "multiple of 128", "fewer tiles than SMs"}
    assert streams == {16, 18, 32}
    # the (width, perms) pairs of -g null rows, c1 (c1 - 1) on both sides of width (width - 1)
    assert {(c[2] > c[1] * (c[1] - 1)) for c in S2_CASES if c[2] is not None} == {True, False}


def test_s2_cases_reach_the_fixed_point_boundaries():
    """F = 48 (the smallest subnormal), -log2 E exactly a power of two (the ib loop's boundary) and M just below 2^56 (all
    entries just above 2^-128), restated on the host from the tables the cases use."""
    got = {}
    cpu = torch.zeros((1, 18), dtype=torch.int16)
    for kind in ("subnormal", "pow2", "near128"):
        e = expected_table(kind, cpu, 18, True, seed=18).numpy()
        mx = float(np.max(-np.log2(e.astype(np.float64))))
        f = fraction_bits(e)
        got[kind] = (f, mx == 2.0 ** round(np.log2(mx)), round(mx * 2.0 ** f) < 2 ** 56 <= round(mx * 2.0 ** f) + 2 ** 30)
    assert got == {"subnormal": (48, False, False), "pow2": (50, True, False), "near128": (49, False, True)}


def test_s1_cases_reach_every_launch():
    """Every launch of launch_s1, and >= 5 groups per warp with a partial last group off CTA 0 for every per-warp-stream
    launch."""
    sms = B200_SMS
    launches, steady = set(), set()
    for k, width, bins, table in S1_CASES:
        name = s1_launch(k, width)
        launches.add(name)
        st = s1_stream(name)
        if st is not None:
            s = k5_schedule(case_bins(bins, sms), *st, sms)
            if s["min_groups"] >= 5 and s["partial"] and s["partial"][0] != 0:
                steady.add(name)
    every = {"direct", "global table", "smem, 1024 threads", "smem, 256 threads x 1 per SM", "smem, 256 threads x 2 per SM",
             "smem, 256 threads x 3 per SM", "smem, 256 threads x 4 per SM"}
    assert launches == every
    assert steady == every - {"direct"}


# ------------------------------------------------------------------------------------------------ GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("case", S2_CASES, ids=[s2_case_id(c) for c in S2_CASES])
def test_s2_scores_on_every_bin(eng, sms, case):
    """Every bin against the float64 reference; the float32-only call is the rounding of the float64 output byte for
    byte and the rounding of the reference but for rare 1-ulp cases; the float64-only call equals the float64 output bit
    for bit; no output is written past either end."""
    k, width, perms, bins_spec, table, rows, mode = case
    bins = case_bins(bins_spec, sms)
    p = width * (width - 1) if perms is None else perms
    cnt = make_counts(bins, k, width, seed=bins * 37 + k * 5 + width, rows=rows)
    e = expected_table(table, cnt, k, True, seed=k * 7 + width)
    assert bool((e == 0).any()) == (table in TABLES_WITH_ZERO)
    route = s2_route(k, width, mode, table in TABLES_WITH_ZERO)
    if route[0] == "tc":
        assert eng.scores_s2_fixed_point(e, k, p)[1] == fraction_bits(e.cpu().numpy())
    check_all_outputs(eng, cnt, width, e, mode, p, s2_reference(cnt, p, e), route, sms)


@pytest.mark.gpu
@pytest.mark.parametrize("k,width,bins_spec,table", S1_CASES,
                         ids=["k%d-w%d-%s-%s" % (k, w, "%dx+%d" % b if b[0] else str(b[1]), t) for k, w, b, t in S1_CASES])
def test_s1_scores_on_every_bin(eng, sms, k, width, bins_spec, table):
    """As the S2 test, for TABLE (every launch of launch_s1) and DIRECT; the two agree bit for bit."""
    bins = case_bins(bins_spec, sms)
    cnt = make_counts(bins, k, width, seed=bins * 41 + k * 3 + width)
    e = expected_table(table, cnt, k, False, seed=k * 11 + width)
    assert bool((e == 0).any()) == (table in TABLES_WITH_ZERO)
    ref = s1_reference(cnt, width, e)
    t32, t64 = check_all_outputs(eng, cnt, width, e, TABLE, None, ref, s1_route(k, width), sms)
    d32, d64 = check_all_outputs(eng, cnt, width, e, DIRECT, None, ref, ("s1", width, "direct"), sms)
    assert_bits_equal(t64, d64, s1_route(k, width), sms, "TABLE vs DIRECT float64")
    assert_bits_equal(t32, d32, s1_route(k, width), sms, "TABLE vs DIRECT float32")


@pytest.mark.gpu
def test_successive_calls_on_one_stream(eng, sms):
    """Calls that change route, state count and table back to back on one stream, with no synchronisation between them:
    each S2 call rebuilds the constant tables, the B operand image and the zero flag in the shared per-device workspace.
    Every output equals its reference and the same call made alone."""
    bins = 128 * 3 * sms + 77
    plan = []
    for name, k, width, table in (("tc", 18, 833, "data"), ("dfma", 18, 2100, "dir4"), ("tc", 18, 833, "zero"),
                                  ("tc", 15, 127, "data"), ("tc", 32, 255, "dir4"), ("s1", 18, 833, "data"),
                                  ("tc", 18, 833, "pow2")):
        cnt = make_counts(bins, k, width, seed=k * 100 + width)
        s2 = name != "s1"
        e = expected_table(table, cnt, k, s2, seed=k + width + len(plan))
        p = width * (width - 1) if s2 else None
        route = s2_route(k, width, TABLE, table in TABLES_WITH_ZERO) if s2 else s1_route(k, width)
        ref = s2_reference(cnt, p, e) if s2 else s1_reference(cnt, width, e)
        plan.append((cnt, width, e, p, route, ref))
    alone = []
    for cnt, width, e, p, route, ref in plan:
        alone.append(call_scores(eng, cnt, width, e, TABLE, p, want64=True, route=route, sms=sms))
        torch.cuda.synchronize()
    seq = [call_scores(eng, cnt, width, e, TABLE, p, want64=True, route=route, sms=sms)
           for cnt, width, e, p, route, ref in plan]
    for (cnt, width, e, p, route, ref), (a32, a64), (s32, s64) in zip(plan, alone, seq):
        assert_f64_close(s64, ref, route, sms)
        assert_bits_equal(s64, a64, route, sms, "float64 output in sequence vs alone")
        assert_bits_equal(s32, a32, route, sms, "float32 output in sequence vs alone")
        assert_f32_rounds_reference(s32, ref, route, sms)


def windows(bins, k, w=4096):
    """Bin ranges at the start, across element 2^31 and byte 2^32 of the float32 output, and at the end."""
    out = [(0, w), (bins - w, bins)]
    for elem in (1 << 30, 1 << 31):                   # 2^30 float32 elements = 2^32 bytes
        b = elem // k
        out.append((b - w // 2, b + w // 2))
    return out


@pytest.mark.gpu
def test_scores_with_64_bit_addressing(eng, sms):
    """bins x K > 2^31 elements (more than 8 GiB of float32 output): the S2 tensor-core kernel and S1 at K = 18, width
    10, and the DFMA S2 kernel at K = 15, width 2100, float32 only.  The reference on bin windows at the start, across
    the 2^31-element and 2^32-byte boundaries and at the end; the whole float32 output against the rounding of a float64
    call's output, in chunks.  About 30 GB of device memory, freed before the test returns."""
    free = torch.cuda.mem_get_info()[0]
    if free < 34 * 2 ** 30:
        pytest.skip("needs about 34 GB of free device memory, %d GB free" % (free >> 30))

    def check(cnt, width, e, perms, route, ref_fn):
        bins, k = cnt.shape
        s32, _ = call_scores(eng, cnt, width, e, TABLE, perms, route=route, sms=sms)
        _, o64 = call_scores(eng, cnt, width, e, TABLE, perms, want32=False, want64=True, route=route, sms=sms)
        for lo, hi in windows(bins, k):
            ref = ref_fn(cnt[lo:hi])
            try:
                assert_f64_close(o64[lo:hi], ref, route, sms)
                assert_f32_rounds_reference(s32[lo:hi], ref, route, sms)
            except AssertionError as err:
                raise AssertionError("window starting at bin %d: %s" % (lo, err))
        step = 1 << 24
        for lo in range(0, bins, step):
            a, b = s32[lo:lo + step], o64[lo:lo + step].to(torch.float32)
            bad = (a.view(torch.int32) != b.view(torch.int32)).nonzero()
            assert not len(bad), "%s: float32 output differs from the rounding of the float64 output at bin %d state %d" % (
                route, lo + int(bad[0, 0]), int(bad[0, 1]))
        del s32, o64
        torch.cuda.empty_cache()

    try:
        k, width = 18, 10
        bins = (1 << 31) // k + 5 * 128 * sms + 77
        cnt = make_counts(bins, k, width, seed=64)
        assert bins * k > 2 ** 31 and bins < 2 ** 31
        e2 = expected_table("dir4", cnt, k, True, seed=1)
        check(cnt, width, e2, width * (width - 1), s2_route(k, width, TABLE, False),
              lambda c: s2_reference(c, width * (width - 1), e2))
        e1 = expected_table("dir4", cnt, k, False, seed=2)
        check(cnt, width, e1, None, s1_route(k, width), lambda c: s1_reference(c, width, e1))
        del cnt
        torch.cuda.empty_cache()
        k, width = 15, 2100
        bins = (1 << 31) // k + 5 * 256 * 3 * sms + 19
        cnt = make_counts(bins, k, width, seed=65)
        e2 = expected_table("dir4", cnt, k, True, seed=3)
        check(cnt, width, e2, width * (width - 1), s2_route(k, width, TABLE, False),
              lambda c: s2_reference(c, width * (width - 1), e2))
        del cnt
    finally:
        torch.cuda.empty_cache()
