"""Text / npz writers of the score stage (scores.py:509-536, 163-169)."""
import ctypes

import numpy as np

from . import _lib


def _gzip_level(level):
    if level is None:
        import os
        level = int(os.environ.get("EPILOGOS_B200_GZIP_LEVEL", "4"))
    return level


def _native_locations(loc):
    """(NUL-separated chromosome names, int32 ids per row, int64 starts, int64 ends) for the native writers."""
    if "chrom_id" in loc:
        cid = np.ascontiguousarray(loc["chrom_id"], dtype=np.int32)
        names = loc["chrom_names"]
    else:
        uniq, cid = np.unique(np.asarray(loc["chrom"], dtype=object).astype(str), return_inverse=True)
        cid = cid.astype(np.int32)
        names = b"\0".join(u.encode() for u in uniq) + b"\0"
    if len(cid) == 0:
        names = names or b"\0"
    return (names, cid, np.ascontiguousarray(loc["start"], dtype=np.int64),
            np.ascontiguousarray(loc["end"], dtype=np.int64))


def write_scores_text(path, scores32, loc, level=None, threads=0):
    """`chr \\t start \\t end \\t K x "{:.5f}"` per bin through gzip (scores.py:530-536), formatted and compressed by
    the native writer (epi_write_scores_gz).  The reference formats np.float32 values with "{:.5f}", i.e. the exact
    binary value rounded to 5 decimals, which is what printf's "%.5f" of the widened double gives.
    `level`: gzip level, default $EPILOGOS_B200_GZIP_LEVEL or 4.  Measured on 1 M rows x 18 scores, 8 vCPUs: level 9 (what
    the reference writes) 0.15 M rows/s, 40.2 MB; 6: 0.86 M rows/s, 41.6 MB; 4: 1.85 M rows/s, 44.4 MB; 1: 2.45 M rows/s,
    51.1 MB -- the decompressed text is the same at any level."""
    level = _gzip_level(level)
    scores32 = np.ascontiguousarray(scores32, dtype=np.float32)
    rows, k = scores32.shape
    names, cid, starts, ends = _native_locations(loc)
    from . import timing
    with timing.stage("format %.5f + deflate"):
        _lib.call("epi_write_scores_gz", str(path).encode(), ctypes.c_char_p(names), ctypes.c_void_p(cid.ctypes.data),
                  ctypes.c_void_p(starts.ctypes.data), ctypes.c_void_p(ends.ctypes.data),
                  ctypes.c_void_p(scores32.ctypes.data), rows, k, int(level), int(threads))


def write_metrics_text(path, loc, state_names, max_diff, distance, pval=None, bh=None, level=None, threads=0):
    """pairwiseMetrics_<tag>.txt.gz through the native writer (epi_write_metrics_gz): per bin `chr \t start \t end \t
    <name of the max-difference state> \t "%.5f" of |distance| \t +/- [\t "%.5e" p \t "%.5e" BH]`."""
    names, cid, starts, ends = _native_locations(loc)
    max_diff = np.ascontiguousarray(max_diff, dtype=np.int32)
    distance = np.ascontiguousarray(distance, dtype=np.float32)
    if (pval is None) != (bh is None):
        raise ValueError("p-values and adjusted p-values go together")
    if pval is not None:
        pval = np.ascontiguousarray(pval, dtype=np.float64)
        bh = np.ascontiguousarray(bh, dtype=np.float64)
    p = lambda a: ctypes.c_void_p(0 if a is None else a.ctypes.data)
    states = b"\0".join(str(n).encode() for n in state_names) + b"\0"
    _lib.call("epi_write_metrics_gz", str(path).encode(), ctypes.c_char_p(names), p(cid), p(starts), p(ends),
              ctypes.c_char_p(states), len(state_names), p(max_diff), p(distance), p(pval), p(bh), len(distance),
              int(_gzip_level(level)), int(threads))


def write_permutations_text(path, loc, k, pval, bh, level=None, threads=0):
    """pairwisePermutation_<tag>.txt.gz through the native writer (epi_write_permutations_gz): per bin `chr \t start \t
    end \t k \t "%.5e" p \t "%.5e" BH`."""
    names, cid, starts, ends = _native_locations(loc)
    k = np.ascontiguousarray(k, dtype=np.uint32)
    pval = np.ascontiguousarray(pval, dtype=np.float64)
    bh = np.ascontiguousarray(bh, dtype=np.float64)
    if not (len(k) == len(pval) == len(bh) == len(starts)):
        raise ValueError("one count, p-value and adjusted p-value per bin")
    p = lambda a: ctypes.c_void_p(a.ctypes.data)
    _lib.call("epi_write_permutations_gz", str(path).encode(), ctypes.c_char_p(names), p(cid), p(starts), p(ends), p(k),
              p(pval), p(bh), len(k), int(_gzip_level(level)), int(threads))


def write_multigroup_text(path, loc, t, group, state, sign, group_names, state_names, k=None, pval=None, bh=None,
                          level=None, threads=0):
    """multigroupMetrics_<tag>.txt.gz through the native writer (epi_write_multigroup_gz): per bin `chr \t start \t end
    \t "%.5e" T \t <driving group> \t <driving state> \t +/- [\t k \t "%.5e" p \t "%.5e" BH]`; group and state are
    0-based indices into group_names and state_names."""
    names, cid, starts, ends = _native_locations(loc)
    t = np.ascontiguousarray(t, dtype=np.float64)
    group = np.ascontiguousarray(group, dtype=np.uint8)
    state = np.ascontiguousarray(state, dtype=np.uint8)
    sign = np.ascontiguousarray(sign, dtype=np.int8)
    if not (len(t) == len(group) == len(state) == len(sign) == len(starts)):
        raise ValueError("one statistic, group, state and sign per bin")
    if not ((k is None) == (pval is None) == (bh is None)):
        raise ValueError("counts, p-values and adjusted p-values go together")
    if k is not None:
        k = np.ascontiguousarray(k, dtype=np.uint32)
        pval = np.ascontiguousarray(pval, dtype=np.float64)
        bh = np.ascontiguousarray(bh, dtype=np.float64)
    p = lambda a: ctypes.c_void_p(0 if a is None else a.ctypes.data)
    gnames = b"\0".join(str(n).encode() for n in group_names) + b"\0"
    states = b"\0".join(str(n).encode() for n in state_names) + b"\0"
    _lib.call("epi_write_multigroup_gz", str(path).encode(), ctypes.c_char_p(names), p(cid), p(starts), p(ends), p(t),
              p(group), p(state), p(sign), ctypes.c_char_p(gnames), len(group_names), ctypes.c_char_p(states),
              len(state_names), p(k), p(pval), p(bh), len(t), int(_gzip_level(level)), int(threads))


def location_array(loc):
    """object [rows, 3] array as produced by pd.read_table(...).to_numpy() in scores.py:161."""
    arr = np.empty((len(loc["chrom"]), 3), dtype=object)
    arr[:, 0] = loc["chrom"]
    arr[:, 1] = loc["start"]
    arr[:, 2] = loc["end"]
    return arr
