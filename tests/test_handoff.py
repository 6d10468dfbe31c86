"""The score stage's hand-over to step 4 (epilogos_b200.handoff) on a stand-in backend: what the temp files carry equals
what the in-memory hand-over carries, in the format the reference and the python -m entry points read."""
import numpy as np
import pytest
import torch

from epilogos_b200 import handoff, roi_pairwise, session, writer
from test_pairwise_stats import StatsBackend

B, K, R = 7, 18, 4            # rows per input file, states, region permutations
TAG = "t"

# The temp files of one input file as a EPILOGOS_B200_KEEP_TEMP=1 run of the command line wrote them before the hand-over
# had one module: (npz key, dtype, shape) in file order.  temp_scores, temp_nullDistances and temp_quiescence are the
# reference's own format.
FORMATS = {
    "temp_scores": (("chrName", "<U4", (1,)), ("scoreArr", "<f4", (B, K)), ("locationArr", "|O", (B, 3))),
    "temp_nullDistances": (("chrName", "<U4", (1,)), ("nullDistances", "<f4", (B,))),
    "temp_quiescence": (("chrName", "<U4", (1,)), ("quiescenceArr", "|b1", (B,))),
    "temp_permutations": (("chrName", "<U4", (1,)), ("exceedances", "<u4", (B,)), ("permutations", "<i8", ())),
    "temp_regionNull": (("chrName", "<U4", (1,)), ("maxima", "<i8", (R,)), ("window", "<i8", ()),
                        ("permutations", "<i8", ())),
    "temp_multigroup": (("chrName", "<U4", (1,)), ("groups", "<U2", (3,)), ("t", "<f8", (B,)), ("group", "|u1", (B,)),
                        ("state", "|u1", (B,)), ("sign", "|i1", (B,)), ("chrom", "<U4", (B,)), ("start", "<i8", (B,)),
                        ("end", "<i8", (B,)), ("exceedances", "<u4", (B,)), ("permutations", "<i8", ())),
}
WITHOUT_PERMUTATIONS = FORMATS["temp_multigroup"][:-2]


def make_record(kind, optional, be, out, name, rng):
    """(record, in_memory) of input file m_<name> as the score stage passes them to publish; paired mode also writes its
    delta text."""
    start = np.arange(B, dtype=np.int64) * 200 + rng.integers(0, 1000) * 200
    loc = dict(chrom=np.array([name] * B, dtype=object), start=start, end=start + 200)
    if kind == "scores":
        return handoff.record(loc, scoreArr=rng.normal(size=(B, K)).astype(np.float32)), None
    extra = {}
    if optional:
        extra = dict(exceedances=torch.from_numpy(rng.integers(0, 4, B).astype(np.int32)), permutations=3,
                     region_maxima=rng.integers(0, 2 ** 40, R).astype(np.int64), region_window=9, region_permutations=R)
    if kind == "paired":
        delta = rng.normal(size=(B, K)).astype(np.float32)
        writer.write_scores_text(out / ("pairwiseDelta_%s_m_%s.txt.gz" % (TAG, name)), delta, loc)
        rec = handoff.record(loc, null=torch.from_numpy(rng.normal(size=B).astype(np.float32)),
                             quiescence=torch.from_numpy((rng.random(B) < 0.3).astype(np.uint8)), **extra)
        return rec, lambda: dict(zip(("distance", "max_diff"),
                                     be.pairwise_real_reduce(torch.from_numpy(delta), text_round_trip=True)))
    return handoff.record(loc, groups=np.array(["g1", "g3", "g5"], dtype=object), t=rng.random(B),
                          group=rng.integers(0, 3, B).astype(np.uint8), state=rng.integers(0, K, B).astype(np.uint8),
                          sign=rng.choice(np.array([-1, 1], dtype=np.int8), B), **extra), None


def expected_files(kind, optional):
    if kind == "scores":
        return {"temp_scores": FORMATS["temp_scores"]}
    if kind == "multigroup":
        files = {"temp_multigroup": FORMATS["temp_multigroup"] if optional else WITHOUT_PERMUTATIONS}
    else:
        files = {p: FORMATS[p] for p in ("temp_nullDistances", "temp_quiescence")}
        if optional:
            files["temp_permutations"] = FORMATS["temp_permutations"]
    if optional:
        files["temp_regionNull"] = FORMATS["temp_regionNull"]
    return files


def collect(kind, out, be):
    if kind == "paired":                 # step 4 completes the file records from the delta text
        return roi_pairwise.readInData(out, TAG, be)
    return handoff.collect(kind, out, TAG)


def host(v):
    return v.numpy() if isinstance(v, torch.Tensor) else v


@pytest.mark.parametrize("kind,optional", [("scores", False), ("paired", False), ("paired", True),
                                           ("multigroup", False), ("multigroup", True)])
def test_temp_files_carry_what_the_hand_over_carries(tmp_path, monkeypatch, kind, optional):
    be = StatsBackend()
    monkeypatch.delenv("EPILOGOS_B200_KEEP_TEMP", raising=False)
    monkeypatch.setattr(session, "handover", {})
    mem, disk = tmp_path / "mem", tmp_path / "disk"
    for out, enabled in ((mem, True), (disk, False)):
        out.mkdir()
        monkeypatch.setattr(session, "handover_enabled", enabled)
        rng = np.random.default_rng(5)
        for name in ("chrX", "chr9"):
            rec, in_memory = make_record(kind, optional, be, out, name, rng)
            handoff.publish(kind, out, TAG, "m_" + name, rec, in_memory=in_memory)
    assert len(session.handover) == 2 and not list(mem.glob("temp_*"))

    files = expected_files(kind, optional)
    assert sorted(f.name for f in disk.glob("temp_*")) == sorted("%s_%s_m_%s.npz" % (p, TAG, c)
                                                                 for p in files for c in ("chrX", "chr9"))
    for f in disk.glob("temp_*"):
        z = np.load(f, allow_pickle=True)
        fmt = tuple((key, z[key].dtype.str, z[key].shape) for key in z.files)
        assert fmt == files[f.name.split("_" + TAG + "_")[0]], f.name

    want, got = collect(kind, mem, be), collect(kind, disk, be)
    assert not session.handover
    assert [c["chrName"] for c in got] == [c["chrName"] for c in want] == ["chr9", "chrX"]
    for g, w in zip(got, want):
        assert sorted(g) == sorted(w)
        for key in w:
            x, y = host(g[key]), host(w[key])
            if isinstance(y, np.ndarray):
                assert x.dtype == y.dtype and x.shape == y.shape and np.array_equal(x, y), key
            else:
                assert type(x) is type(y) and x == y, key
        if "exceedances" in w:
            assert isinstance(w["exceedances"], np.ndarray) and w["exceedances"].dtype == np.uint32

    other = disk / ("%s_other_m_chr1.npz" % next(iter(files)))
    other.write_bytes(b"")
    handoff.remove_temps(kind, disk, TAG)
    # single mode removes every temp_scores file of the directory, whatever its tag, as the reference's roiSingle does
    assert sorted(f.name for f in disk.glob("temp_*")) == ([] if kind == "scores" else [other.name])


def test_nothing_to_collect_is_an_error(tmp_path):
    with pytest.raises(FileNotFoundError, match="temp_multigroup_t_"):
        handoff.collect("multigroup", tmp_path, TAG)
