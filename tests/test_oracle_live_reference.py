"""The CPU oracle against the UNMODIFIED reference run now, on inputs that are in no fixture.

tests/test_oracle_golden.py pins the oracle to committed outputs of the reference; this module draws fresh matrices (seeded,
so a failure can be replayed) and runs the reference itself -- expected.main -> expectedCombination.main -> scores.main
through oracle/reference_driver.py -- wherever it can be imported (the checkout EPILOGOS_REFERENCE names, or the
byte-compiled oracle/_ref that __graft_entry__.build() stages from it).  Skipped where neither exists.  Same bar as the fixtures:
integer tables, float32 expected payload, float32 scores, formatted text and seeded null distances bit for bit.
"""
import numpy as np
import pytest

from oracle import epilogos_oracle as orc
from oracle import reference_driver as ref

pytestmark = [pytest.mark.skipif(not ref.available(), reason="the reference is neither named by EPILOGOS_REFERENCE nor staged in oracle/_ref"),
              pytest.mark.filterwarnings("ignore:This process .* is multi-threaded, use of fork:DeprecationWarning")]   # its Pool


def _matrix(rng, bins, cols, k, kind):
    if kind == "uniform":
        return rng.integers(0, k, size=(bins, cols)).astype(np.int8)
    x = rng.integers(0, k, size=(bins, cols)).astype(np.int8)
    dominant = rng.integers(0, k, size=(bins, 1))
    x = np.where(rng.random((bins, cols)) < 0.7, dominant, x).astype(np.int8)
    x[: bins // 10] = k - 1                                        # an all-quiescent stretch: zeros in the S2 / S3 tables
    return x


@pytest.mark.parametrize("seed,bins,cols,k,kind,nproc", [(20261017, 240, 37, 18, "realistic", 1), (20261018, 151, 64, 15, "uniform", 3),
                                                         (20261019, 97, 9, 25, "realistic", 2)])
def test_single_mode_s1_s2_fresh_inputs(seed, bins, cols, k, kind, nproc):
    rng = np.random.default_rng(seed)
    x = _matrix(rng, bins, cols, k, kind)
    starts = np.arange(bins) * 200
    for s in (1, 2):
        r = ref.run_single(x, k, s, nproc=nproc)
        counts = orc.s1_expected_counts(x, k) if s == 1 else orc.s2_expected_counts(x, k)
        assert counts.dtype == r["counts"].dtype and np.array_equal(counts, r["counts"])
        exp = orc.normalize_expected(counts)
        assert exp.dtype == r["exp"].dtype and exp.tobytes() == r["exp"].tobytes()
        scores = orc.s1_scores(x, k, exp) if s == 1 else orc.s2_scores(x, k, exp)
        assert scores.tobytes() == r["scores"].tobytes()
        assert orc.format_scores_text(scores, "chr1", starts, starts + 200) == r["scores_text"]
        rowloop = orc.s1_scores_rowloop(x, k, exp) if s == 1 else orc.s2_scores_rowloop(x, k, exp)
        assert rowloop.tobytes() == r["scores"].tobytes()


def test_single_mode_s3_fresh_input():
    rng = np.random.default_rng(20261020)
    bins, cols, k = 60, 7, 6
    x = _matrix(rng, bins, cols, k, "realistic")
    r = ref.run_single(x, k, 3)
    n3 = orc.s3_expected_counts(x, k)
    assert np.array_equal(n3, r["counts"]) and int(n3.sum()) == bins * cols * (cols - 1)
    e3 = orc.normalize_expected(n3)
    assert e3.tobytes() == r["exp"].tobytes()
    assert orc.s3_scores_rowloop(x, k, e3).tobytes() == r["scores"].tobytes()
    assert np.max(np.abs(orc.s3_scores_f64(x, k, e3) - r["scores"])) < 1e-4      # 42 pair terms per bin: float32 noise only


@pytest.mark.parametrize("seed,c1,c2,k,group_size,quiescent", [(20261021, 13, 9, 18, -1, None), (20261022, 20, 17, 15, 8, 0)])
def test_paired_mode_fresh_inputs(seed, c1, c2, k, group_size, quiescent):
    rng = np.random.default_rng(seed)
    bins = 180
    xa, xb = _matrix(rng, bins, c1, k, "realistic"), _matrix(rng, bins, c2, k, "realistic")
    q = k - 1 if quiescent is None else quiescent
    comb = np.concatenate((xa, xb), axis=1)
    perm = orc.reference_shuffle_indices(seed, bins, c1 + c2)
    starts = np.arange(bins) * 200
    for s in (1, 2):
        r = ref.run_paired(xa, xb, k, s, seed, quiescent_state=q, group_size=group_size)
        counts = orc.s1_expected_counts(comb, k) if s == 1 else orc.s2_expected_counts(comb, k)
        assert np.array_equal(counts, r["counts"])
        exp = orc.normalize_expected(counts)
        assert exp.tobytes() == r["exp"].tobytes()
        o = orc.paired_scores(xa, xb, perm, k, s, exp, q, group_size)
        assert np.array_equal(o["quiescence"], r["quiescence"])
        assert o["null_distances"].tobytes() == r["null_distances"].tobytes()
        assert orc.format_scores_text(o["delta"], "chr1", starts, starts + 200) == r["delta_text"]
