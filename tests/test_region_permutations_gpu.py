"""Region-null kernels (csrc/label_permutations.cu) against numpy: epi_split_counts over states, widths, group counts,
tails and unaligned matrices, its identity split against epi_group_counts, its rejected bitsets; epi_window_max over
windows, dtypes, chunking and its input range; and the CLI end to end against the numpy oracle (tests/region_oracle.py)
with the identity split reproducing the observed statistic."""
import numpy as np
import pytest

import region_oracle as ro

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from epilogos_b200 import build, engine
    build.build()
    engine.device_info()
    return engine


def matrix(rng, bins, N, K, kind):
    if kind == "uniform":
        return rng.integers(0, K, size=(bins, N)).astype(np.int8)
    x = np.full((bins, N), K - 1, dtype=np.int8)                  # mostly quiescent, a few states per bin
    for b in range(bins):
        if rng.random() < 0.6:
            states = rng.choice(K, size=min(K, 1 + rng.integers(0, 4)), replace=False)
            x[b] = rng.choice(states, size=N)
    return x


def random_members(rng, nsplit, N, sizes):
    """Bitsets [nsplit, G - 1, words] of random splits with group sizes `sizes`, and the splits' column groups."""
    G = len(sizes)
    words = (N + 63) // 64
    edges = np.cumsum([0] + list(sizes))
    bits = np.zeros((nsplit, G - 1, words * 64), dtype=np.uint8)
    groups = []
    for p in range(nsplit):
        perm = rng.permutation(N)
        groups.append([perm[edges[g]:edges[g + 1]] for g in range(G)])
        for g in range(G - 1):
            bits[p, g, groups[-1][g]] = 1
    return np.packbits(bits, axis=2, bitorder="little").view(np.uint64), groups


def device_matrix(x, pad, offset):
    """x on the device with row pitch N + pad and a base `offset` bytes past a 256-byte boundary."""
    bins, N = x.shape
    pitch = N + pad
    buf = torch.zeros(offset + bins * pitch + 16, dtype=torch.int8)
    host = buf[offset:offset + bins * pitch].view(bins, pitch)
    host[:, :N] = torch.from_numpy(x)
    dev = buf.cuda()
    return dev[offset:offset + bins * pitch].view(bins, pitch)


def sizes_for(N, G, rng):
    cut = np.sort(rng.integers(0, N + 1, size=G - 1))
    return list(np.diff(np.concatenate(([0], cut, [N]))))


CASES = [(15, 833, 2, "realistic"), (18, 833, 3, "uniform"), (25, 65, 2, "uniform"), (32, 64, 64, "uniform"),
         (18, 63, 3, "realistic"), (18, 1, 2, "uniform"), (32, 65535, 3, "uniform"), (15, 65535, 2, "realistic"),
         (18, 833, 64, "realistic"), (25, 200, 3, "realistic")]


@pytest.mark.parametrize("K,N,G,kind", CASES)
def test_split_counts_against_numpy(eng, K, N, G, kind):
    from oracle import epilogos_oracle as orc
    rng = np.random.default_rng(K * 1000 + N + G)
    bins = 37 if N > 5000 else 101                               # not a multiple of the 32-bin tile
    nsplit = 11                                                  # not a multiple of the 8 warps
    x = matrix(rng, bins, N, K, kind)
    sizes = sizes_for(N, G, rng)
    members, groups = random_members(rng, nsplit, N, sizes)
    xd = device_matrix(x, pad=3, offset=5)                       # unaligned pitch and base
    cnt = eng.split_counts(xd, N, K, torch.from_numpy(members.view(np.int64)).cuda(), G)
    got = cnt.cpu().numpy().view(np.uint16)
    for p in range(nsplit):
        for g in range(G):
            assert cnt[p, g].data_ptr() % 16 == 0
            want = orc.bin_counts(x[:, np.sort(groups[p][g])], K) if len(groups[p][g]) else np.zeros((bins, K))
            assert np.array_equal(got[p, g], want), (p, g)


def test_identity_split_equals_group_counts(eng):
    rng = np.random.default_rng(3)
    x = matrix(rng, 1000, 833, 18, "realistic")
    xd = eng.pack_states(x).cuda()
    words = (833 + 63) // 64
    bits = np.zeros((1, 1, words * 64), dtype=np.uint8)
    bits[0, 0, :400] = 1
    members = torch.from_numpy(np.packbits(bits, axis=2, bitorder="little").view(np.int64)).cuda()
    cnt = eng.split_counts(xd, 833, 18, members, 2)
    want = eng.group_counts(xd, 833, 18, [range(400), range(400, 833)])
    assert torch.equal(cnt[0, 0], want[0]) and torch.equal(cnt[0, 1], want[1])
    assert torch.equal(cnt[0, 0] + cnt[0, 1], eng.bin_counts(xd, 833, 18))


def test_rejected_bitsets(eng):
    from epilogos_b200 import _lib
    x = eng.pack_states(np.zeros((10, 70), dtype=np.int8)).cuda()
    m = np.zeros((2, 2, 2), dtype=np.uint64)
    m[1, 0, 0] = 0b1100
    m[1, 1, 0] = 0b0100                                          # column 2 in two groups of split 1
    with pytest.raises(_lib.EpilogosB200Error, match="split 1: group 1 shares column 2"):
        eng.split_counts(x, 70, 18, torch.from_numpy(m.view(np.int64)).cuda(), 3)
    m = np.zeros((1, 1, 2), dtype=np.uint64)
    m[0, 0, 1] = np.uint64(1) << np.uint64(8)                    # column 72 >= cols = 70
    with pytest.raises(_lib.EpilogosB200Error, match="column 72, at or above cols=70"):
        eng.split_counts(x, 70, 18, torch.from_numpy(m.view(np.int64)).cuda(), 2)


def np_window_max(vals, W):
    return np.array([ro.window_max(ro.q(v), W) for v in vals], dtype=np.int64)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("W", [1, 2, 125, 16384])
def test_window_max_against_numpy(eng, dtype, W):
    rng = np.random.default_rng(W)
    for n in (W - 1, W, W + 1, 3 * 4096 + W + 17):
        if n < 0:
            continue
        vals = (rng.random((3, n)) ** 4 * 50).astype(np.float32 if dtype == torch.float32 else np.float64)
        vals[:, ::7] = 0
        init = torch.tensor([-1, 5, 2 ** 60], dtype=torch.int64, device="cuda")
        got = eng.window_max(torch.from_numpy(vals).cuda(), W, init.clone()).cpu().numpy()
        want = np.maximum(np_window_max(vals, W), init.cpu().numpy()) if n >= W else init.cpu().numpy()
        assert got.tolist() == want.tolist(), n
        if n > 2 * W:                                            # chunks overlapping by W - 1 equal one call
            m = torch.full((3,), -1, dtype=torch.int64, device="cuda")
            d = torch.from_numpy(vals).cuda()
            cut = n // 2
            eng.window_max(d[:, :cut + W - 1].contiguous(), W, m)
            eng.window_max(d[:, cut:].contiguous(), W, m)
            assert m.cpu().numpy().tolist() == np_window_max(vals, W).tolist()


def test_window_max_input_range(eng):
    from epilogos_b200 import _lib
    top32, top64 = np.nextafter(np.float32(2 ** 24), np.float32(0)), np.nextafter(2.0 ** 24, 0)
    for dtype, top in ((torch.float32, top32), (torch.float64, top64)):
        v = torch.tensor([[0.0, -0.0, float(top)]], dtype=dtype, device="cuda")
        m = eng.window_max(v, 3, torch.full((1,), -1, dtype=torch.int64, device="cuda"))
        assert int(m.item()) == int(np.rint(np.float64(top) * 2 ** 24))
        for bad in (2.0 ** 24, float("nan"), float("inf"), -float("inf"), -1e-3):
            v = torch.tensor([[1.0, 2.0], [3.0, bad]], dtype=dtype, device="cuda")
            with pytest.raises(_lib.EpilogosB200Error, match=r"stat\[1\]\[1\]"):
                eng.window_max(v, 2, torch.zeros(2, dtype=torch.int64, device="cuda"))


def test_identity_split_maxima_equal_the_observed_window_maximum(eng, monkeypatch):
    """With split 0 replaced by the identity, the backend's maximum for it is the largest window sum of the real
    statistic the stages compute (paired: |distance| of the real delta after the text round trip; multi-group: T)."""
    from epilogos_b200 import region_null
    from epilogos_b200.backend import CudaBackend
    be = CudaBackend()
    rng = np.random.default_rng(8)
    N, K, W = 300, 18, 125
    x = matrix(rng, 5000, N, K, "realistic")
    xd = eng.pack_states(x).cuda()
    real_blocks = region_null.split_blocks

    def with_identity(seed, sizes, nperm, block):
        for p0, m in real_blocks(seed, sizes, nperm, block):
            if p0 == 0:
                bits = np.zeros((N,), dtype=np.uint8)
                m = m.copy()
                edges = np.cumsum([0] + list(sizes))
                for g in range(len(sizes) - 1):
                    bits[:] = 0
                    bits[edges[g]:edges[g + 1]] = 1
                    m[0, g] = np.packbits(np.concatenate([bits, np.zeros(m.shape[2] * 64 - N, np.uint8)]),
                                          bitorder="little").view(np.uint64)
            yield p0, m
    monkeypatch.setattr(region_null, "split_blocks", with_identity)
    for saliency in (1, 2):
        for sizes in ((140, 160), (100, 90, 110)):
            edges = np.cumsum([0] + list(sizes))
            cnt = eng.group_counts(xd, N, K, [range(edges[g], edges[g + 1]) for g in range(len(sizes))])
            union = eng.bin_counts(xd, N, K)
            n1, n2 = eng.expected_tables(union, N, want_s1=saliency == 1, want_s2=saliency == 2)
            exp = eng.normalize(n1 if saliency == 1 else n2)
            if len(sizes) == 2:
                sa = be.scores(cnt[0].clone(), sizes[0], saliency, exp, perms=sizes[0] * (sizes[0] - 1))
                sb = be.scores(cnt[1].clone(), sizes[1], saliency, exp, perms=sizes[1] * (sizes[1] - 1))
                delta, _ = be.pairwise_combine(sa, sb, None, None)
                real = be.pairwise_real_reduce(delta, text_round_trip=True)[0].abs()
                m = be.region_maxima_paired(xd, None, sizes, K, W, 5, 99, saliency, exp, workspace_bytes=1 << 22)
            else:
                real = be.multigroup_stat(cnt, list(sizes), saliency, exp)[0]
                m = be.region_maxima_multigroup(xd, None, sizes, K, W, 5, 99, saliency, exp, workspace_bytes=1 << 22)
            want = ro.window_max(ro.q(real.cpu().numpy()), W)
            assert int(m[0].item()) == want, (saliency, sizes)
            assert np.all(m[1:].cpu().numpy() >= 0)


def test_maxima_do_not_depend_on_the_workspace_or_a_halo(eng):
    """Two workspace caps, and the rows split in two with the second part passed as host halo rows of the first part's
    call (the rows mode of several ranks), give the same maxima."""
    from epilogos_b200.backend import CudaBackend
    be = CudaBackend()
    rng = np.random.default_rng(4)
    N, K, W = 120, 15, 50
    x = matrix(rng, 3000, N, K, "uniform")
    xd = eng.pack_states(x).cuda()
    union = eng.bin_counts(xd, N, K)
    n1, _ = eng.expected_tables(union, N, want_s1=True, want_s2=False)
    exp = eng.normalize(n1)
    args = ((50, 70), K, W, 9, 5, 1, exp)
    a = be.region_maxima_paired(xd, None, *args, workspace_bytes=1 << 30)
    b = be.region_maxima_paired(xd, None, *args, workspace_bytes=1 << 18)
    assert torch.equal(a, b)
    cut = 1700
    first = be.region_maxima_paired(eng.pack_states(x[:cut]).cuda(), x[cut:cut + W - 1], *args)
    second = be.region_maxima_paired(eng.pack_states(x[cut:]).cuda(), None, *args)
    assert torch.equal(torch.maximum(first, second), a)


@pytest.mark.parametrize("saliency", [1, 2])
def test_cli_end_to_end_against_the_oracle(eng, tmp_path, monkeypatch, saliency):
    """Paired (-a/-b) and multi-group runs on the GPU write the region files of the numpy oracle's stand-in backend; the
    S2 paired run uses the reference null mode, whose scores are the reference's float64 expression."""
    from click.testing import CliRunner
    from epilogos_b200 import run, session
    from test_cli import META
    from test_host_stages import write_tsv
    from test_region_permutations import RegionBackend
    rng = np.random.default_rng(5)
    a, b, inp = tmp_path / "a", tmp_path / "b", tmp_path / "in"
    for d in (a, b, inp):
        d.mkdir()
    for chrom, rows in (("chr1", 700), ("chr2", 411)):
        x = matrix(rng, rows, 60, 18, "realistic")
        x[: rows // 4, :25] = rng.integers(0, 3, size=(rows // 4, 25))
        write_tsv(a / ("m_%s.txt.gz" % chrom), x[:, :25], chrom=chrom, gz=True)
        write_tsv(b / ("m_%s.txt.gz" % chrom), x[:, 25:], chrom=chrom, gz=True)
        write_tsv(inp / ("m_%s.txt.gz" % chrom), x, chrom=chrom, gz=True)
    meta = tmp_path / "meta.tsv"
    meta.write_text(META)
    gfile = tmp_path / "g.tsv"
    gfile.write_text("p\t1-20\nq\t21-38\nr\t39-60\n")
    monkeypatch.setenv("EPILOGOS_B200_SEED", "19")
    if saliency == 2:
        monkeypatch.setenv("EPILOGOS_B200_NULL", "reference")

    def cli(out, backend, *args):
        session.clear()
        if backend is not None:
            monkeypatch.setattr(session, "_backend", backend)
        r = CliRunner().invoke(run.main, ["-j", str(meta), "-s", str(saliency), "-w", "50", "-o", str(out),
                                          "--roi-permutations", "64"] + list(args))
        session.clear()
        monkeypatch.setattr(session, "_backend", None)
        assert r.exit_code == 0 and r.exception is None, r.output + repr(r.exception)

    runs = [(["-m", "paired", "-a", str(a), "-b", str(b)], "", "a_b_s%d" % saliency)]
    if saliency == 1:
        runs.append((["-m", "paired", "-i", str(inp), "--groups", str(gfile), "--multigroup", "p,q,r"], "p_q_r",
                     "p_q_r_s1"))
    for args, sub, tag in runs:
        cli(tmp_path / "gpu", None, *args)
        cli(tmp_path / "numpy", RegionBackend(), *args)
        for name in ("regionPermutation_%s.txt" % tag, "regionsOfInterest_%s.txt" % tag):
            got = (tmp_path / "gpu" / sub / name).read_text()
            assert got == (tmp_path / "numpy" / sub / name).read_text(), name
        zg = np.load(tmp_path / "gpu" / sub / ("regionNullMaxima_%s.npz" % tag))
        zn = np.load(tmp_path / "numpy" / sub / ("regionNullMaxima_%s.npz" % tag))
        assert zg["maxima"].tolist() == zn["maxima"].tolist() and int(zg["permutations"]) == 64
        reg = (tmp_path / "gpu" / sub / ("regionPermutation_%s.txt" % tag)).read_text()
        k = [int(r.split("\t")[4]) for r in reg.splitlines()]
        assert len(k) > 0 and max(k) <= 64
