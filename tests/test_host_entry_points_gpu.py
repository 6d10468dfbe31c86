"""The host-buffer entry points of csrc/pipeline.cu at the sizes the benchmark runs them.

epi_single_host / epi_single_host_packed copy the matrix in chunks and alternate between two device buffers; from chunk 2
on a buffer is reused behind the events of the chunk before last.  The cases here run four to six chunks with a partial
last chunk, the 4,096-bin minimum chunk, every host layout (packed, pinned int8 in the device pitch, pageable int8 at
pitch == cols) and a sequence of calls that grows and then reuses the cached buffers.  epi_paired_host draws its null
shuffles in batches; the paired cases run three batches, and two shards whose batch sizes differ from the whole call's.

chunk_bins and null_batch restate the chunk and batch sizes of csrc/pipeline.cu; every case asserts how many chunks or
batches it runs.  References: int64 tables summed from integer products of the device counts, orc.normalize_expected,
the device-level entry points on a device copy of the whole matrix (no chunks, no batches), the float64 oracle on a
sample of bins, and the numpy restatement of the shuffle sampler (tests/sampler_oracle.py).
"""
import numpy as np
import pytest

import sampler_oracle as so

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import epilogos_oracle as orc            # noqa: E402  (checker only)

RTOL, ATOL = 1e-9, 1e-12
MARGIN, MAX_EXCLUDED = 1e-8, 10       # draws this close to a cumulative boundary may differ (test_sampler_gpu.py)


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import build, engine
    build.build()
    engine.device_info()
    return engine


def u16(cnt):
    """int16 tensor holding uint16 counts -> int64 tensor of the counts."""
    return cnt.to(torch.int64) & 0xffff


def chunk_bins(bins, cols):
    """Bins per H2D chunk of single_host_impl: ~192 MiB of rows in the device pitch, a multiple of 4,096 bins, at least
    4,096, at most the matrix."""
    dpitch = (cols + 15) & ~15
    return min(bins, max(4096, (192 << 20) // dpitch // 4096 * 4096))


def null_batch(bins, k, nperm):
    """Permutations per null batch of epi_paired_host: ~256 MiB of float32 scores per group, at least 1, at most nperm."""
    return max(1, min(nperm, (256 << 20) // (bins * k * 4)))


def batch_sizes(n, size):
    return [min(size, n - lo) for lo in range(0, n, size)]


def oracle_counts(x, idx, cols, k, block=256):
    """orc.bin_counts of the rows idx of a host matrix, a block of rows at a time."""
    return np.concatenate([orc.bin_counts(x[idx[lo:lo + block], :cols], k) for lo in range(0, len(idx), block)])


def exact_tables(cnt, block=1 << 20):
    """(n1 int64 [K], n2 int64 [K, K]) of uint16 counts [bins, K] on the device, in int64: n1 = sum_b c, n2[s] = sum_b
    c[s] c - [s = t] n1."""
    k = cnt.shape[1]
    n1 = torch.zeros(k, dtype=torch.int64, device=cnt.device)
    n2 = torch.zeros((k, k), dtype=torch.int64, device=cnt.device)
    for lo in range(0, cnt.shape[0], block):
        c = u16(cnt[lo:lo + block])
        n1 += c.sum(dim=0)
        for s in range(k):
            n2[s] += (c[:, s:s + 1] * c).sum(dim=0)
    n2 -= torch.diag(n1)
    return n1.cpu().numpy(), n2.cpu().numpy()


# ------------------------------------------------------------------------------------------------ single matrix
def device_states(bins, cols, k, seed):
    """int8 [bins, pitch_for(cols)] on the device.  Per bin a dominant state holds a random share of the labels (scores
    from flat to peaked), the rest are uniform; the first and the last bin of every 4,096 bins (so of every chunk) hold
    one state throughout.  Pad bytes are 7 and never interpreted."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    pitch = (cols + 15) & ~15
    x = torch.full((bins, pitch), 7, dtype=torch.int8, device="cuda")
    rows = max(1, (1 << 25) // cols)
    for lo in range(0, bins, rows):
        n = min(rows, bins - lo)
        other = torch.randint(0, k, (n, cols), generator=g, device="cuda", dtype=torch.int8)
        dom = torch.randint(0, k, (n, 1), generator=g, device="cuda", dtype=torch.int8)
        share = torch.rand((n, 1), generator=g, device="cuda")
        keep = torch.rand((n, cols), generator=g, device="cuda") < share
        x[lo:lo + n, :cols] = torch.where(keep, dom, other)
        del other, keep
    first = torch.arange(0, bins, 4096, device="cuda")
    last = torch.clamp(first + 4095, max=bins - 1)
    x[first, :cols] = (first % k).to(torch.int8)[:, None].expand(-1, cols)
    x[last, :cols] = ((last * 7 + 3) % k).to(torch.int8)[:, None].expand(-1, cols)
    return x


def host_inputs(eng, x, cols, k, kinds):
    """The host layouts of the device matrix x: 'int8' pinned in the device pitch (one contiguous copy per chunk),
    'dense' pageable with pitch == cols (cudaMemcpy2DAsync), 'packed' pinned 4 / 5-bit transport layout."""
    xh = torch.empty(x.shape, dtype=torch.int8, pin_memory=True)
    xh.copy_(x)
    out = {"int8": xh}
    if "dense" in kinds:
        out["dense"] = np.ascontiguousarray(xh.numpy()[:, :cols])
    if "packed" in kinds:
        out["packed"] = eng.pack_bits_host(xh, cols, k)
        assert out["packed"][1] == (4 if k <= 16 else 5)
    return out


def run_host(eng, kind, data, cols, k, saliency, want_scores=True):
    """One host call; the scores are copied out of the cached pinned buffer they alias."""
    if kind == "packed":
        packed, bits = data
        counts, exp, scores = eng.single_host_packed(packed, cols, k, saliency, bits, want_scores=want_scores)
    else:
        counts, exp, scores = eng.single_host(data, cols, k, saliency, want_scores=want_scores)
    return counts, exp, None if scores is None else scores.copy()


class SingleReference:
    """What a host call on the matrix x must return: the device-level entry points on the whole device matrix, and int64
    tables from integer products of its counts."""

    def __init__(self, eng, x, cols, k):
        self.eng, self.cols, self.k = eng, cols, k
        self.cnt = eng.bin_counts(x, cols, k)
        self.n = dict(zip((1, 2), exact_tables(self.cnt)))
        n1, n2 = eng.expected_tables(self.cnt, cols)
        assert np.array_equal(n1.cpu().numpy(), self.n[1]) and np.array_equal(n2.cpu().numpy(), self.n[2])
        self.tables = {1: n1, 2: n2}

    def device_path(self, saliency):
        """(exp on the device, float32 scores [bins, K] as numpy): normalize -> scores in TABLE mode."""
        e = self.eng.normalize(self.tables[saliency])
        assert e.cpu().numpy().tobytes() == orc.normalize_expected(self.n[saliency]).tobytes()
        if saliency == 1:
            s = self.eng.scores_s1(self.cnt, self.cols, e)
        else:
            s = self.eng.scores_s2(self.cnt, self.cols, e)
        return e, s.cpu().numpy()

    def check_call(self, saliency, got, want_scores, chunk, what):
        counts, exp, scores = got
        assert np.array_equal(counts, self.n[saliency]), "%s: count table" % what
        assert exp.tobytes() == orc.normalize_expected(self.n[saliency]).tobytes(), "%s: expected table" % what
        if want_scores is None:
            assert scores is None
            return
        bad = np.flatnonzero((scores.view(np.uint32) != want_scores.view(np.uint32)).any(axis=1))
        if len(bad):
            b = int(bad[0])
            c = b // chunk
            raise AssertionError("%s: %d of %d bins differ from the device-level path; the first is bin %d, row %d of chunk %d "
                                 "(buffer %d; chunks with a difference: %s): %s, want %s"
                                 % (what, len(bad), len(scores), b, b - c * chunk, c, c & 1,
                                    sorted(set((bad // chunk).tolist())), scores[b].tolist(), want_scores[b].tolist()))

    def check_sample(self, xh, saliency, e, idx, scores):
        """On the bins idx: K1 counts against orc.bin_counts, the device's float64 scores against the float64 oracle, and
        the host call's float32 scores equal to their rounding."""
        cols, k = self.cols, self.k
        cd = self.cnt[torch.from_numpy(idx).cuda()]
        c = u16(cd).cpu().numpy()
        assert np.array_equal(c, oracle_counts(xh, idx, cols, k))
        en = e.cpu().numpy()
        if saliency == 1:
            _, s64 = self.eng.scores_s1(cd, cols, e, want64=True)
            ref = orc.s1_scores_from_counts(c, cols, en, np.float64)
        else:
            _, s64 = self.eng.scores_s2(cd, cols, e, want64=True)
            ref = orc.s2_scores_from_counts(c, cols * (cols - 1), en, np.float64)
        np.testing.assert_allclose(s64.cpu().numpy(), ref, rtol=RTOL, atol=ATOL)
        assert scores[idx].tobytes() == s64.to(torch.float32).cpu().numpy().tobytes()


def sample_bins(bins, chunk, rng, edge=64, n=2000):
    """The first and last `edge` bins of every chunk and n random bins."""
    parts = [rng.choice(bins, size=min(n, bins), replace=False)]
    for lo in range(0, bins, chunk):
        hi = min(lo + chunk, bins)
        parts += [np.arange(lo, min(lo + edge, hi)), np.arange(max(hi - edge, lo), hi)]
    return np.unique(np.concatenate(parts))


def shape(cols, chunks, last):
    """(bins, bins per chunk) of a matrix of `chunks` chunks whose last one holds `last` bins."""
    chunk = chunk_bins(1 << 40, cols)
    bins = (chunks - 1) * chunk + last
    assert 0 < last < chunk and chunk_bins(bins, cols) == chunk and -(-bins // chunk) == chunks
    return bins, chunk


SINGLE = [  # cols, K, chunks, bins in the last chunk, host layouts
    (833, 18, 6, 1001, ("packed", "int8", "dense")),      # 233,472 bins per chunk
    (127, 15, 4, 77, ("packed", "int8")),                 # 1,572,864 bins per chunk
    (49153, 18, 4, 5, ("int8", "dense")),                 # the 4,096-bin minimum; S1 at this width takes the DIRECT path
]                                                         # (packed rows this long exceed the unpack kernel's shared memory)


def test_single_host_call_sequence_grows_and_reuses_its_buffers(eng):
    """Four calls in a row, each against its own fresh reference.  The second (more bins) grows the count and score
    buffers; the third is the first packed call, at a width whose packed chunk (24,576 rows of 5,120 bytes) is larger
    than one of the other two widths, so it grows the packed buffers unless an earlier call in the process needed more;
    the fourth runs the first shape again on another matrix, with every buffer larger than it needs."""
    calls = [  # cols, K, chunks, bins in the last chunk, layout, saliency
        (833, 18, 6, 1001, "int8", 2),
        (127, 15, 4, 77, "int8", 1),
        (8191, 18, 4, 5, "packed", 2),
        (833, 18, 6, 1001, "packed", 1),
    ]
    pbuf = [chunk_bins(1 << 40, c) * eng.packed_pitch(c, eng.packed_bits(k)) for c, k in ((833, 18), (127, 15), (8191, 18))]
    assert pbuf[2] > max(pbuf[:2])
    for i, (cols, k, nchunks, last, kind, saliency) in enumerate(calls):
        bins, chunk = shape(cols, nchunks, last)
        x = device_states(bins, cols, k, seed=1000 + i)
        inputs = host_inputs(eng, x, cols, k, (kind,))
        ref = SingleReference(eng, x, cols, k)
        del x
        _, want = ref.device_path(saliency)
        got = run_host(eng, kind, inputs[kind], cols, k, saliency)
        ref.check_call(saliency, got, want, chunk, "call %d: %s S%d, %d bins x %d columns" % (i + 1, kind, saliency, bins,
                                                                                            cols))
        print("call %d: c%d k%d %s S%d, %d chunks of %d bins" % (i + 1, cols, k, kind, saliency, nchunks, chunk))
        del ref, inputs, want, got
        torch.cuda.empty_cache()


@pytest.mark.parametrize("case", SINGLE, ids=lambda c: "c%d_k%d_%dchunks" % c[:3])
def test_single_host_over_many_chunks(eng, case):
    """Every layout, S1 and S2: the tables exactly, exp byte for byte, the float32 scores of every bin bit-identical to
    the device-level path (so the layouts agree with each other), the sample against the oracle, and the same tables
    without scores."""
    cols, k, nchunks, last, kinds = case
    bins, chunk = shape(cols, nchunks, last)
    x = device_states(bins, cols, k, seed=cols * 100 + k)
    inputs = host_inputs(eng, x, cols, k, kinds)
    ref = SingleReference(eng, x, cols, k)
    del x
    idx = sample_bins(bins, chunk, np.random.default_rng(cols))
    xh = inputs["int8"].numpy()
    for saliency in (1, 2):
        e, want = ref.device_path(saliency)
        for kind in kinds:
            what = "%s S%d, %d bins x %d columns" % (kind, saliency, bins, cols)
            got = run_host(eng, kind, inputs[kind], cols, k, saliency)
            ref.check_call(saliency, got, want, chunk, what)
            ref.check_call(saliency, run_host(eng, kind, inputs[kind], cols, k, saliency, want_scores=False), None,
                           chunk, what + ", no scores")
        ref.check_sample(xh, saliency, e, idx, got[2])
        del e, want, got
    print("single host c%d k%d: %d bins, %d chunks of %d bins (last %d), layouts %s, S1 and S2, %d sampled bins"
          % (cols, k, bins, nchunks, chunk, last, "/".join(kinds), len(idx)))
    del ref, inputs
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ paired
C1, C2, PK = 12, 9, 18
P1, P2 = C1 * (C1 - 1), C2 * (C2 - 1)      # the S2 normalisers of the real groups, also used for the shuffled ones
BLOCK = 333_334                             # the matrix is a block of rows and two row permutations of it
NPERM = 7
SEED = 0xC0FFEE1500000000 | 0x2A
OFFSET = (1 << 33) + 5
GROUP_SIZES = [-1, 8]


@pytest.fixture(scope="module")
def paired(eng):
    """1,000,002 bins of 12 + 9 biosamples: a block of synthetic rows followed by two row permutations of it, so the
    count tables of the first block, of the other two and of the whole are proportional and their expected tables equal
    (each is the same quotient of exact integers).  Oracle tables and quiescence mask of the whole matrix."""
    base = orc.synth_states(BLOCK, C1 + C2, PK, seed=21)
    rng = np.random.default_rng(21)
    x = np.concatenate([base, base[rng.permutation(BLOCK)], base[rng.permutation(BLOCK)]])
    xa, xb = x[:, :C1], x[:, C1:]
    out = dict(x=x, ha=eng.pack_states(xa), hb=eng.pack_states(xb), bins=len(x),
               n={1: orc.s1_expected_counts(x, PK), 2: orc.s2_expected_counts(x, PK)},
               quiescent=orc.quiescent_mask(xa, xb, PK - 1), runs={})
    assert 0 < out["quiescent"].sum() < len(x)
    yield out
    out.clear()
    torch.cuda.empty_cache()


def paired_call(eng, pd, saliency, group_size, lo=0, hi=None):
    """epi_paired_host on rows [lo, hi) (bin_offset OFFSET + lo), cached per argument set; outputs copied to numpy."""
    key = (saliency, group_size, lo, hi)
    if key not in pd["runs"]:
        hi = pd["bins"] if hi is None else hi
        r = eng.paired_host(pd["ha"][lo:hi], C1, pd["hb"][lo:hi], C2, PK, saliency, PK - 1, group_size=group_size,
                            seed=SEED, bin_offset=OFFSET + lo, nperm=NPERM)
        pd["runs"][key] = {name: np.array(v) for name, v in r.items()}
    return pd["runs"][key]


def device_paired(eng, pd, saliency, group_size):
    """The production paired path on the device copies of the whole matrix: K1 on both groups, the union's table, scores
    at the groups' widths, delta, quiescence mask, and null row p = permutation p of shuffled_counts_philox_range drawn
    on its own, scored at the shuffled widths with the real groups' S2 normalisers, combined."""
    from epilogos_b200.pairwise import shuffled_widths
    size_a, size_b = shuffled_widths(C1, C2, group_size)
    ca, cb = eng.bin_counts(pd["ha"].cuda(), C1, PK), eng.bin_counts(pd["hb"].cuda(), C2, PK)
    cc = (u16(ca) + u16(cb)).to(torch.int16)
    n1, n2 = eng.expected_tables(cc, C1 + C2)
    e = eng.normalize(n1 if saliency == 1 else n2)

    def score(c, width, perms, want64=False):
        if saliency == 1:
            return eng.scores_s1(c, max(width, 1), e, want64=want64)
        return eng.scores_s2(c, max(width, 1), e, perms=perms, want64=want64)

    delta, _ = eng.pairwise_combine(score(ca, C1, P1), score(cb, C2, P2))
    null = []
    for p in range(NPERM):
        oa, ob = eng.shuffled_counts_philox_range(ca, cb, size_a, size_b, SEED, p, 1, C1 + C2, bin_offset=OFFSET)
        _, nd = eng.pairwise_combine(null_a=score(oa[0], size_a, P1), null_b=score(ob[0], size_b, P2))
        null.append(nd.cpu().numpy())
        del oa, ob
    return dict(ca=ca, cb=cb, e=e, score=score, n=(n1 if saliency == 1 else n2).cpu().numpy(),
                delta=delta.cpu().numpy(), quiescent=eng.quiescent_mask(ca, C1, cb, C2, PK - 1).cpu().numpy() == 1,
                null=np.stack(null))


@pytest.mark.parametrize("saliency", [1, 2])
def test_paired_host_outputs_on_a_multi_batch_shape(eng, paired, saliency):
    """counts, exp, delta and the quiescence mask of a call with three null batches: equal to the device-level path on
    every bin and to the oracle (tables and mask of every bin; counts and float64 scores on a sample)."""
    bins = paired["bins"]
    assert batch_sizes(NPERM, null_batch(bins, PK, NPERM)) == [3, 3, 1]
    r = paired_call(eng, paired, saliency, -1)
    d = device_paired(eng, paired, saliency, -1)
    want_n = paired["n"][saliency]
    assert np.array_equal(r["counts"], want_n) and np.array_equal(d["n"], want_n)
    assert r["exp"].tobytes() == orc.normalize_expected(want_n).tobytes() == d["e"].cpu().numpy().tobytes()
    assert r["delta"].tobytes() == d["delta"].tobytes()
    assert np.array_equal(r["quiescent"], paired["quiescent"]) and np.array_equal(d["quiescent"], paired["quiescent"])
    idx = np.unique(np.concatenate([np.random.default_rng(saliency).choice(bins, 2000, replace=False),
                                    np.arange(64), np.arange(bins - 64, bins)]))
    x, en = paired["x"][idx], r["exp"]
    ca, cb = orc.bin_counts(x[:, :C1], PK), orc.bin_counts(x[:, C1:], PK)
    ti = torch.from_numpy(idx).cuda()
    sa, sb = d["ca"][ti], d["cb"][ti]
    assert np.array_equal(u16(sa).cpu().numpy(), ca) and np.array_equal(u16(sb).cpu().numpy(), cb)
    _, a64 = d["score"](sa, C1, P1, want64=True)
    _, b64 = d["score"](sb, C2, P2, want64=True)
    if saliency == 1:
        ra, rb = orc.s1_scores_from_counts(ca, C1, en, np.float64), orc.s1_scores_from_counts(cb, C2, en, np.float64)
    else:
        ra, rb = orc.s2_scores_from_counts(ca, P1, en, np.float64), orc.s2_scores_from_counts(cb, P2, en, np.float64)
    np.testing.assert_allclose(a64.cpu().numpy(), ra, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(b64.cpu().numpy(), rb, rtol=RTOL, atol=ATOL)
    delta = a64.to(torch.float32).cpu().numpy() - b64.to(torch.float32).cpu().numpy()
    assert r["delta"][idx].tobytes() == delta.tobytes()


@pytest.mark.parametrize("group_size", GROUP_SIZES)
@pytest.mark.parametrize("saliency", [1, 2])
def test_paired_host_null_rows_are_the_production_draws(eng, paired, saliency, group_size):
    """Null row p of a call that draws permutations in batches of 3, 3 and 1 equals, byte for byte, permutation p of
    shuffled_counts_philox_range for the same seed and global bins, scored and combined as the production path does."""
    batch = null_batch(paired["bins"], PK, NPERM)
    assert batch_sizes(NPERM, batch) == [3, 3, 1]
    r = paired_call(eng, paired, saliency, group_size)
    want = device_paired(eng, paired, saliency, group_size)["null"]
    assert r["null"].shape == want.shape == (NPERM, paired["bins"])
    for p in range(NPERM):
        bad = np.flatnonzero(r["null"][p].view(np.uint32) != want[p].view(np.uint32))
        assert not len(bad), ("null row %d (batch %d, permutation %d of it): %d of %d bins differ from permutation %d of "
                              "the stream, the first at bin %d: %r, want %r"
                              % (p, p // batch, p % batch, len(bad), paired["bins"], p, bad[0], r["null"][p][bad[0]],
                                 want[p][bad[0]]))
    print("paired S%d g%d: %d null rows in batches %s" % (saliency, group_size, NPERM, batch_sizes(NPERM, batch)))


@pytest.mark.parametrize("group_size", GROUP_SIZES)
@pytest.mark.parametrize("saliency", [1, 2])
def test_paired_host_does_not_depend_on_sharding(eng, paired, saliency, group_size):
    """The whole call against the first block and the rest with their global bin offsets.  The three calls batch the
    permutations differently (3+3+1, 7, 5+2); with equal expected tables every per-bin output of the two shards,
    concatenated, equals the whole call's byte for byte."""
    bins, h = paired["bins"], BLOCK
    sizes = [batch_sizes(NPERM, null_batch(n, PK, NPERM)) for n in (bins, h, bins - h)]
    assert sizes == [[3, 3, 1], [7], [5, 2]]
    whole = paired_call(eng, paired, saliency, group_size)
    first = paired_call(eng, paired, saliency, group_size, 0, h)
    rest = paired_call(eng, paired, saliency, group_size, h, bins)
    assert np.array_equal(whole["counts"], 3 * first["counts"]) and np.array_equal(rest["counts"], 2 * first["counts"])
    assert whole["exp"].tobytes() == first["exp"].tobytes() == rest["exp"].tobytes()
    for name in ("delta", "quiescent"):
        assert np.concatenate([first[name], rest[name]]).tobytes() == whole[name].tobytes(), name
    null = np.concatenate([first["null"], rest["null"]], axis=1)
    bad = np.argwhere(null.view(np.uint32) != whole["null"].view(np.uint32))
    assert not len(bad), "%d nulls differ between the sharded and the whole call, the first at (permutation, bin) %s" % (
        len(bad), bad[0].tolist())
    print("paired S%d g%d sharded at %d: batches %s" % (saliency, group_size, h, sizes))


def null_bounds(a, b):
    """float64 scores a, b [M, K] of the two shuffled groups -> (null, tol, sure): null = sum_s d_s^2 sign(sum_s d_s),
    d = a - b, in float64.  The device has float32 scores within the score tolerance of a and b and one rounding away,
    rounds d_s, the squares and the partial sums to float32; tol bounds what that does to null (twice the rounding unit
    throughout), and sure marks the rows whose sign(sum_s d_s) it cannot flip."""
    u = 2.0 ** -23
    ea = (u + RTOL) * np.abs(a) + ATOL
    eb = (u + RTOL) * np.abs(b) + ATOL
    d = a - b
    ed = ea + eb + u * (np.abs(d) + ea + eb)
    k = a.shape[1]
    sq = np.sum(d * d, axis=1)
    esq = np.sum(ed * (2 * np.abs(d) + ed), axis=1)
    tol = esq + k * u * (sq + esq)
    s = np.sum(d, axis=1)
    sure = np.abs(s) > np.sum(ed, axis=1) + k * u * np.sum(np.abs(d) + ed, axis=1)
    return sq * np.sign(s), tol, sure


@pytest.mark.parametrize("group_size", GROUP_SIZES)
@pytest.mark.parametrize("saliency", [1, 2])
def test_paired_host_nulls_against_the_restated_sampler(eng, paired, saliency, group_size):
    """100 bins of every permutation (so of every batch): the shuffle drawn by the numpy restatement from the oracle's
    counts, scored by the float64 oracle and combined in float64, within the float32 error of the call's null distance.
    Bins with a draw within 1e-8 of a cumulative boundary are left out (expected none)."""
    from epilogos_b200.pairwise import shuffled_widths
    size_a, size_b = shuffled_widths(C1, C2, group_size)
    bins, x = paired["bins"], paired["x"]
    r = paired_call(eng, paired, saliency, group_size)
    rng = np.random.default_rng(saliency * 100 + group_size)
    perm = np.repeat(np.arange(NPERM), 100)
    b = np.concatenate([rng.choice(bins, 100, replace=False) for _ in range(NPERM)])
    ca, cb = orc.bin_counts(x[b, :C1], PK), orc.bin_counts(x[b, C1:], PK)
    dr = so.draw_shuffle(SEED, perm, OFFSET + b, ca, cb, size_a, size_b)
    exp = orc.normalize_expected(paired["n"][saliency])
    assert r["exp"].tobytes() == exp.tobytes()
    if saliency == 1:
        na = orc.s1_scores_from_counts(dr["a"], max(size_a, 1), exp, np.float64)
        nb = orc.s1_scores_from_counts(dr["b"], max(size_b, 1), exp, np.float64)
    else:
        na = orc.s2_scores_from_counts(dr["a"], P1, exp, np.float64)
        nb = orc.s2_scores_from_counts(dr["b"], P2, exp, np.float64)
    null, tol, sure = null_bounds(na, nb)
    got = r["null"][perm, b].astype(np.float64)
    ok = np.where(sure, np.abs(got - null) <= tol, (got == 0) | (np.abs(np.abs(got) - np.abs(null)) <= tol))
    near = ((dr["ma"] <= MARGIN) | (dr["mb"] <= MARGIN)).any(axis=1)
    assert near.sum() <= MAX_EXCLUDED
    bad = np.flatnonzero(~ok & ~near)
    assert not len(bad), ("%d of %d nulls outside the float32 error of the restatement, the first permutation %d bin %d: "
                          "%r, want %r +- %g" % (len(bad), len(b), perm[bad[0]], b[bad[0]], got[bad[0]], null[bad[0]],
                                                 tol[bad[0]]))
    assert np.count_nonzero(null) > len(b) // 2
    print("paired S%d g%d: %d nulls against the restated sampler, %d left out near a boundary, %d with an uncertain sign"
          % (saliency, group_size, len(b) - near.sum(), near.sum(), (~sure).sum()))
