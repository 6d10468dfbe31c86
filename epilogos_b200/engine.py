"""Thin torch-tensor wrappers over the C ABI (include/epilogos_b200.h).

torch is used for device memory, streams and (in the stage drivers) torch.distributed only; every
computation below is a call into libepilogos_b200.so.  All functions raise if the library or a B200 is
missing -- there is no CPU path.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import EPI_SCORE_DIRECT, EPI_SCORE_TABLE  # noqa: F401

S1_TABLE_MAX_WIDTH = 4095      # widest score width of the S1 value table (csrc/common.cuh)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _seed(seed):
    """A Python integer seed as the library's uint64 (taken modulo 2^64)."""
    return ctypes.c_uint64(int(seed) & (2 ** 64 - 1))


def _require_cuda(t, dtype, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.is_contiguous()):
        raise TypeError("%s must be a contiguous CUDA tensor of dtype %s" % (name, dtype))


def pitch_for(cols):
    """Row pitch (bytes) of the packed state matrix: next multiple of 16 (TMA global stride rule)."""
    return (int(cols) + 15) & ~15


def pack_states(states0, pin=True):
    """0-based integer state matrix [bins, C] (any int dtype, numpy) -> pinned int8 [bins, pitch] torch tensor.
    Mirrors the tail of helpers.readStates (helpers.py:154-155: labels - 1, here narrowed to int8).
    Pad bytes are zero and never interpreted."""
    a = np.asarray(states0)
    if a.ndim != 2:
        raise ValueError("state matrix must be 2-D [bins, biosamples]")
    if a.size and (a.min() < 0 or a.max() >= _lib.EPI_MAX_STATES):
        raise ValueError("state labels must be in [0, %d)" % _lib.EPI_MAX_STATES)
    bins, cols = a.shape
    out = torch.zeros((bins, pitch_for(cols)), dtype=torch.int8, pin_memory=bool(pin and torch.cuda.is_available()))
    out.numpy()[:, :cols] = a
    return out


def bin_counts(x, cols, num_states, out=None):
    """K1.  x: CUDA int8 [bins, pitch]; returns CUDA int16 tensor [bins, K] holding uint16 counts."""
    _require_cuda(x, torch.int8, "x")
    bins, pitch = x.shape
    if out is None:
        out = torch.empty((bins, num_states), dtype=torch.int16, device=x.device)
    _lib.call("epi_bin_counts", _ptr(x), bins, int(cols), pitch, int(num_states), _ptr(out), _stream())
    return out


def group_counts(x, cols, num_states, groups):
    """Counts of column groups of one matrix, read once.  x: CUDA int8 [bins, pitch]; groups: sequences of 0-based column
    indices.  Returns CUDA int16 [len(groups), bins, K] holding uint16 counts; block g is bin_counts of group g's columns."""
    _require_cuda(x, torch.int8, "x")
    bins, pitch = x.shape
    lists = [np.asarray(g, dtype=np.int32).ravel() for g in groups]
    offsets = np.concatenate(([0], np.cumsum([len(g) for g in lists]))).astype(np.int32)
    flat = torch.from_numpy(np.concatenate(lists) if lists else np.zeros(0, np.int32)).to(x.device)
    offs = torch.from_numpy(offsets).to(x.device)
    out = torch.empty((len(lists), bins, num_states), dtype=torch.int16, device=x.device)
    _lib.call("epi_group_counts", _ptr(x), bins, int(cols), pitch, int(num_states), _ptr(flat), _ptr(offs), len(lists),
              _ptr(out), _stream())
    return out


def gather_columns(x, cols, idx):
    """The columns idx (0-based, in the given order) of x (CUDA int8 [bins, pitch]) as a new CUDA int8
    [bins, pitch_for(len(idx))] matrix with zero pad bytes."""
    _require_cuda(x, torch.int8, "x")
    bins, pitch = x.shape
    idx_dev = torch.from_numpy(np.asarray(idx, dtype=np.int32).ravel()).to(x.device)
    n = idx_dev.numel()
    out = torch.empty((bins, pitch_for(max(n, 1))), dtype=torch.int8, device=x.device)
    _lib.call("epi_gather_columns", _ptr(x), bins, int(cols), pitch, _ptr(idx_dev), n, _ptr(out), out.shape[1], _stream())
    return out


def expected_tables(cnt, width, want_s1=True, want_s2=True):
    """K2.  Returns (n1 int64[K] or None, n2 int64[K,K] or None) for this shard."""
    _require_cuda(cnt, torch.int16, "cnt")
    bins, k = cnt.shape
    n1 = torch.zeros(k, dtype=torch.int64, device=cnt.device) if want_s1 else None
    n2 = torch.zeros((k, k), dtype=torch.int64, device=cnt.device) if want_s2 else None
    _lib.call("epi_expected_s1s2", _ptr(cnt), bins, k, int(width), _ptr(n1), _ptr(n2), _stream())
    return n1, n2


def normalize(counts):
    """K4.  int64 count table -> float32 probabilities (expectedCombination.py:42)."""
    _require_cuda(counts, torch.int64, "counts")
    out = torch.empty(counts.shape, dtype=torch.float32, device=counts.device)
    _lib.call("epi_normalize_i64", _ptr(counts), counts.numel(), _ptr(out), _stream())
    return out


def scores_s1(cnt, width, exp1, want64=False, mode=EPI_SCORE_TABLE, out32=None):
    _require_cuda(cnt, torch.int16, "cnt")
    _require_cuda(exp1, torch.float32, "exp1")
    bins, k = cnt.shape
    if exp1.numel() != k:
        raise ValueError("expected table has %d entries, need %d" % (exp1.numel(), k))
    if out32 is None:
        out32 = torch.empty((bins, k), dtype=torch.float32, device=cnt.device)
    out64 = torch.empty((bins, k), dtype=torch.float64, device=cnt.device) if want64 else None
    _lib.call("epi_scores_s1", _ptr(cnt), bins, k, int(width), _ptr(exp1), _ptr(out32), _ptr(out64), int(mode),
              _stream())
    return (out32, out64) if want64 else out32


def scores_s2(cnt, width, exp2, perms=None, want64=False, mode=EPI_SCORE_TABLE, out32=None):
    _require_cuda(cnt, torch.int16, "cnt")
    _require_cuda(exp2, torch.float32, "exp2")
    bins, k = cnt.shape
    if exp2.numel() != k * k:
        raise ValueError("expected table has %d entries, need %d" % (exp2.numel(), k * k))
    if perms is None:
        perms = int(width) * (int(width) - 1)
    if out32 is None:
        out32 = torch.empty((bins, k), dtype=torch.float32, device=cnt.device)
    out64 = torch.empty((bins, k), dtype=torch.float64, device=cnt.device) if want64 else None
    _lib.call("epi_scores_s2", _ptr(cnt), bins, k, int(width), int(perms), _ptr(exp2), _ptr(out32), _ptr(out64),
              int(mode), _stream())
    return (out32, out64) if want64 else out32


def scores_s2_fixed_point(exp2, num_states, perms):
    """(M int64 tensor [K, K] on the device, F): M = round(-log2 E2 * 2^F), the 56-bit fixed-point table (seven base-256
    digits, F = 56 - ib with -log2 E2 < 2^ib) that the tensor-core S2 scores multiply the counts with."""
    _require_cuda(exp2, torch.float32, "exp2")
    m = torch.empty((num_states, num_states), dtype=torch.int64, device=exp2.device)
    f = ctypes.c_int32(0)
    _lib.call("epi_scores_s2_fixed_point", _ptr(exp2), int(num_states), int(perms), _ptr(m), ctypes.byref(f), _stream())
    return m, f.value


_pinned_scores = {}


def single_host(x_host, cols, num_states, saliency, want_scores=True, scores_out=None):
    """Whole S1/S2 path on a HOST matrix (numpy int8 [bins, pitch] or a pinned torch int8 tensor).
    Returns (counts int64 ndarray, exp float32 ndarray, scores float32 ndarray or None).  `scores_out` may be a
    pinned float32 torch tensor [bins, K] to receive the scores; otherwise one pinned buffer per shape is kept and
    reused (the returned array aliases it until the next call with the same shape)."""
    if isinstance(x_host, torch.Tensor):
        if x_host.is_cuda or x_host.dtype != torch.int8 or not x_host.is_contiguous():
            raise TypeError("x_host must be a contiguous CPU int8 tensor")
        bins, pitch = x_host.shape
        xp = ctypes.c_void_p(x_host.data_ptr())
    else:
        x_host = np.ascontiguousarray(x_host, dtype=np.int8)
        bins, pitch = x_host.shape
        xp = ctypes.c_void_p(x_host.ctypes.data)
    shape = (num_states,) if saliency == 1 else (num_states, num_states)
    counts = np.empty(shape, dtype=np.int64)
    exp = np.empty(shape, dtype=np.float32)
    scores = None
    sp = ctypes.c_void_p(0)
    if want_scores:
        if scores_out is None:
            key = (bins, num_states)
            if key not in _pinned_scores:
                _pinned_scores.clear()
                _pinned_scores[key] = torch.empty((bins, num_states), dtype=torch.float32, pin_memory=True)
            scores_out = _pinned_scores[key]
        if scores_out.dtype != torch.float32 or tuple(scores_out.shape) != (bins, num_states):
            raise TypeError("scores_out must be a float32 tensor of shape [bins, K]")
        scores = scores_out.numpy()
        sp = ctypes.c_void_p(scores_out.data_ptr())
    _lib.call("epi_single_host", xp, bins, int(cols), pitch, int(num_states), int(saliency),
              ctypes.c_void_p(counts.ctypes.data), ctypes.c_void_p(exp.ctypes.data), sp)
    return counts, exp, scores


# ------------------------------------------------------------------------------------------------ packed transport layout
def packed_bits(num_states):
    return int(_lib.load().epi_packed_bits(int(num_states)))


def packed_pitch(cols, bits):
    return int(_lib.load().epi_packed_pitch(int(cols), int(bits)))


def pack_bits_host(x_host, cols, num_states, out=None, threads=0):
    """int8 host matrix [bins, pitch] (numpy or CPU torch tensor) -> bit-packed host matrix uint8 [bins, packed_pitch]
    (pinned when a GPU is present), 4 bits per label for <= 16 states, else 5.  Runs on CPU threads; no GPU needed."""
    if isinstance(x_host, torch.Tensor):
        xp, (bins, pitch) = ctypes.c_void_p(x_host.data_ptr()), x_host.shape
    else:
        x_host = np.ascontiguousarray(x_host, dtype=np.int8)
        xp, (bins, pitch) = ctypes.c_void_p(x_host.ctypes.data), x_host.shape
    bits = packed_bits(num_states)
    pp = packed_pitch(cols, bits)
    if out is None:
        out = torch.empty((bins, pp), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    _lib.call("epi_pack_states_host", xp, bins, int(cols), pitch, bits, ctypes.c_void_p(out.data_ptr()), pp, int(threads))
    return out, bits


def pack_bits(x, cols, num_states):
    """Device int8 [bins, pitch] -> device packed uint8 [bins, packed_pitch]."""
    _require_cuda(x, torch.int8, "x")
    bits = packed_bits(num_states)
    pp = packed_pitch(cols, bits)
    out = torch.empty((x.shape[0], pp), dtype=torch.uint8, device=x.device)
    _lib.call("epi_pack_states", _ptr(x), x.shape[0], int(cols), x.shape[1], bits, _ptr(out), pp, _stream())
    return out, bits


def unpack_bits(packed, cols, bits):
    """Device packed uint8 [bins, packed_pitch] -> device int8 [bins, pitch_for(cols)] (pad bytes beyond the last group
    of 8 labels are not written)."""
    _require_cuda(packed, torch.uint8, "packed")
    out = torch.zeros((packed.shape[0], pitch_for(cols)), dtype=torch.int8, device=packed.device)
    _lib.call("epi_unpack_states", _ptr(packed), packed.shape[0], int(cols), int(bits), packed.shape[1], _ptr(out),
              out.shape[1], _stream())
    return out


def single_host_packed(packed_host, cols, num_states, saliency, bits, want_scores=True, scores_out=None):
    """single_host with the matrix in the bit-packed transport layout (CPU uint8 tensor [bins, packed_pitch])."""
    if packed_host.is_cuda or packed_host.dtype != torch.uint8 or not packed_host.is_contiguous():
        raise TypeError("packed_host must be a contiguous CPU uint8 tensor")
    bins, pp = packed_host.shape
    shape = (num_states,) if saliency == 1 else (num_states, num_states)
    counts = np.empty(shape, dtype=np.int64)
    exp = np.empty(shape, dtype=np.float32)
    scores, sp = None, ctypes.c_void_p(0)
    if want_scores:
        if scores_out is None:
            key = (bins, num_states)
            if key not in _pinned_scores:
                _pinned_scores.clear()
                _pinned_scores[key] = torch.empty((bins, num_states), dtype=torch.float32, pin_memory=True)
            scores_out = _pinned_scores[key]
        scores, sp = scores_out.numpy(), ctypes.c_void_p(scores_out.data_ptr())
    _lib.call("epi_single_host_packed", ctypes.c_void_p(packed_host.data_ptr()), bins, int(cols), pp, int(bits),
              int(num_states), int(saliency), ctypes.c_void_p(counts.ctypes.data), ctypes.c_void_p(exp.ctypes.data), sp)
    return counts, exp, scores


def s3_host(x_host, cols, num_states, want_exp=True, scores_out=None):
    """Whole S3 path on a HOST matrix (CPU int8 torch tensor [bins, pitch]): (exp float32 [C,C,K,K] or None, scores)."""
    bins, pitch = x_host.shape
    exp = np.empty((cols, cols, num_states, num_states), dtype=np.float32) if want_exp else None
    if scores_out is None:
        scores_out = torch.empty((bins, num_states), dtype=torch.float32, pin_memory=True)
    _lib.call("epi_s3_host", ctypes.c_void_p(x_host.data_ptr()), bins, int(cols), pitch, int(num_states),
              ctypes.c_void_p(exp.ctypes.data if want_exp else 0), ctypes.c_void_p(scores_out.data_ptr()))
    return exp, scores_out.numpy()


def paired_host(xa_host, cols_a, xb_host, cols_b, num_states, saliency, quiescent_state, group_size=-1, seed=0,
                bin_offset=0, nperm=1, null_out=None, delta_out=None):
    """Paired mode on HOST matrices (CPU int8 torch tensors).  Returns dict(counts, exp, delta, null [nperm, bins], quiescent)."""
    bins = xa_host.shape[0]
    shape = (num_states,) if saliency == 1 else (num_states, num_states)
    counts = np.empty(shape, dtype=np.int64)
    exp = np.empty(shape, dtype=np.float32)
    if delta_out is None:
        delta_out = torch.empty((bins, num_states), dtype=torch.float32, pin_memory=True)
    if null_out is None:
        null_out = torch.empty((max(nperm, 1), bins), dtype=torch.float32, pin_memory=True)
    quies = np.empty(bins, dtype=np.uint8)
    _lib.call("epi_paired_host", ctypes.c_void_p(xa_host.data_ptr()), xa_host.shape[1], int(cols_a),
              ctypes.c_void_p(xb_host.data_ptr()), xb_host.shape[1], int(cols_b), bins, int(num_states), int(saliency),
              int(quiescent_state), int(group_size), _seed(seed), int(bin_offset), int(nperm),
              ctypes.c_void_p(counts.ctypes.data), ctypes.c_void_p(exp.ctypes.data), ctypes.c_void_p(delta_out.data_ptr()),
              ctypes.c_void_p(null_out.data_ptr() if nperm > 0 else 0), ctypes.c_void_p(quies.ctypes.data))
    return dict(counts=counts, exp=exp, delta=delta_out.numpy(), null=null_out.numpy()[:nperm], quiescent=quies.astype(bool))


def device_info():
    sm, major, minor = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0)
    _lib.call("epi_device_info", ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor))
    return dict(sm_count=sm.value, cc=(major.value, minor.value))


def counts_to_numpy(cnt):
    """CUDA int16 storage of uint16 counts -> numpy uint16."""
    return cnt.cpu().numpy().view(np.uint16)


# ------------------------------------------------------------------------------------------------ S3
def s3_plan(bins, cols, num_states):
    vals = [ctypes.c_int64(0) for _ in range(5)]
    _lib.call("epi_s3_plan", int(bins), int(cols), int(num_states), *[ctypes.byref(v) for v in vals])
    mp, bp, ntiles, onehot_bytes, tile_bytes = [v.value for v in vals]
    return dict(mp=mp, bp=bp, ntiles=ntiles, onehot_bytes=onehot_bytes, tile_bytes=tile_bytes)


S3_CHUNK_BINS = 131072      # bins per Gram launch: keeps the ~148 tiles in flight in lock-step on their L2 panels


def s3_expected_tiles(x, cols, num_states, tiles=None, onehot_budget_bytes=None, chunk_bins=None):
    """K3.  x: CUDA int8 [bins, pitch].  Returns (tiles int32 tensor, plan): the upper-triangular 128x256 tiles of
    the one-hot Gram matrix of this shard (the quantity that is all-reduced across ranks).  Bins are processed
    in chunks so that the transposed one-hot workspace stays below `onehot_budget_bytes`."""
    _require_cuda(x, torch.int8, "x")
    bins, pitch = x.shape
    plan = s3_plan(bins, cols, num_states)
    mp = plan["mp"]
    if tiles is None:
        tiles = torch.empty(plan["tile_bytes"] // 4, dtype=torch.int32, device=x.device)
    chunk = chunk_bins or S3_CHUNK_BINS
    if onehot_budget_bytes is not None:
        chunk = min(chunk, (onehot_budget_bytes // mp) // 128 * 128)
    chunk = max(128, min(plan["bp"], chunk // 128 * 128))
    oht = torch.empty(mp * min(chunk, plan["bp"]), dtype=torch.int8, device=x.device)
    first = True
    for lo in range(0, bins, chunk):
        n = min(chunk, bins - lo)
        bp = (n + 127) // 128 * 128
        xs = x[lo:lo + n]
        _lib.call("epi_s3_onehot", _ptr(xs), n, int(cols), pitch, int(num_states), _ptr(oht), mp, bp, _stream())
        _lib.call("epi_s3_gram", _ptr(oht), mp, bp, _ptr(tiles), 0 if first else 1, _stream())
        first = False
    if first:      # no bins at all
        tiles.zero_()
    return tiles, plan


def s3_finalize(tiles, cols, num_states, mp, total_bins, want_counts=True, want_exp=True):
    """Tile buffer (after the all-reduce) -> (counts int64 [C,C,K,K] or None, exp float32 [C,C,K,K] or None)."""
    _require_cuda(tiles, torch.int32, "tiles")
    shape = (cols, cols, num_states, num_states)
    counts = torch.empty(shape, dtype=torch.int64, device=tiles.device) if want_counts else None
    exp = torch.empty(shape, dtype=torch.float32, device=tiles.device) if want_exp else None
    _lib.call("epi_s3_finalize", _ptr(tiles), int(cols), int(num_states), int(mp), int(total_bins), _ptr(counts),
              _ptr(exp), _stream())
    return counts, exp


def s3_terms(exp3, cols, num_states):
    """float32 expected table [C,C,K,K] -> float64 pair terms q*log2(q/E) (scores.py:479-480)."""
    _require_cuda(exp3, torch.float32, "exp3")
    if exp3.numel() != cols * cols * num_states * num_states:
        raise ValueError("expected table has %d entries, need %d" % (exp3.numel(), cols * cols * num_states ** 2))
    n = ctypes.c_int64(0)
    _lib.call("epi_s3_terms_size", int(cols), int(num_states), ctypes.byref(n))
    terms = torch.empty(n.value, dtype=torch.float64, device=exp3.device)
    _lib.call("epi_s3_terms", _ptr(exp3), int(cols), int(num_states), _ptr(terms), _stream())
    return terms


def s3_terms_dense(terms, cols, num_states):
    """View of the padded term blocks as a dense [C, C, K, K] tensor (copies)."""
    kk = num_states * num_states
    blk = (kk + 1) & ~1
    return terms[: cols * cols * blk].reshape(cols * cols, blk)[:, :kk].reshape(cols, cols, num_states, num_states)


def scores_s3(x, cols, num_states, terms, want64=False, out32=None):
    """K6.  x: CUDA int8 [bins, pitch]; terms from s3_terms()."""
    _require_cuda(x, torch.int8, "x")
    _require_cuda(terms, torch.float64, "terms")
    bins, pitch = x.shape
    if out32 is None:
        out32 = torch.empty((bins, num_states), dtype=torch.float32, device=x.device)
    out64 = torch.empty((bins, num_states), dtype=torch.float64, device=x.device) if want64 else None
    _lib.call("epi_scores_s3", _ptr(x), bins, int(cols), pitch, int(num_states), _ptr(terms), _ptr(out32), _ptr(out64),
              _stream())
    return (out32, out64) if want64 else out32


# ------------------------------------------------------------------------------------------------ paired
def shuffled_counts_perm(xa, cols_a, xb, cols_b, perm, num_states, size_a, size_b):
    """Counts of the shuffled halves A', B' for explicit permutation indices (int32 [bins, cols_a+cols_b])."""
    _require_cuda(xa, torch.int8, "xa")
    _require_cuda(xb, torch.int8, "xb")
    _require_cuda(perm, torch.int32, "perm")
    bins = xa.shape[0]
    ca = torch.empty((bins, num_states), dtype=torch.int16, device=xa.device)
    cb = torch.empty((bins, num_states), dtype=torch.int16, device=xa.device)
    _lib.call("epi_shuffled_counts_perm", _ptr(xa), xa.shape[1], int(cols_a), _ptr(xb), xb.shape[1], int(cols_b),
              _ptr(perm), bins, int(num_states), int(size_a), int(size_b), _ptr(ca), _ptr(cb), _stream())
    return ca, cb


def shuffled_counts_philox(cnt_a, cnt_b, size_a, size_b, seed, nperm=1, width=None, bin_offset=0):
    """nperm uniform shuffles per bin drawn on the device; returns int16 tensors [nperm, bins, K].
    `width` = combined number of biosamples (default: size_a + size_b, right unless -g shrinks the groups);
    `bin_offset` = global index of row 0 (the random stream of a bin is keyed by its global index)."""
    return shuffled_counts_philox_range(cnt_a, cnt_b, size_a, size_b, seed, 0, nperm,
                                        width if width is not None else size_a + size_b, bin_offset)


def shuffled_counts_philox_range(cnt_a, cnt_b, size_a, size_b, seed, perm_offset, nperm, width, bin_offset=0):
    """shuffled_counts_philox for permutations perm_offset .. perm_offset + nperm - 1: int16 tensors [nperm, bins, K]."""
    _require_cuda(cnt_a, torch.int16, "cnt_a")
    _require_cuda(cnt_b, torch.int16, "cnt_b")
    bins, k = cnt_a.shape
    oa = torch.empty((nperm, bins, k), dtype=torch.int16, device=cnt_a.device)
    ob = torch.empty((nperm, bins, k), dtype=torch.int16, device=cnt_a.device)
    _lib.call("epi_shuffled_counts_philox_range", _ptr(cnt_a), _ptr(cnt_b), bins, k, int(width), int(size_a), int(size_b),
              _seed(seed), int(bin_offset), int(perm_offset), int(nperm), _ptr(oa), _ptr(ob), _stream())
    return oa, ob


def null_exceedances(null_a, null_b, dist, k):
    """k[b] += #{p : |null distance of (null_a[p, b], null_b[p, b])| >= |dist[b]|}.  null_a, null_b: float32 score arrays
    [nperm, bins, K]; dist: float32 [bins]; k: int32 [bins] holding uint32 counts (updated in place)."""
    _require_cuda(null_a, torch.float32, "null_a")
    _require_cuda(null_b, torch.float32, "null_b")
    _require_cuda(dist, torch.float32, "dist")
    _require_cuda(k, torch.int32, "k")
    nperm, bins, K = null_a.shape
    if tuple(null_b.shape) != (nperm, bins, K) or dist.numel() != bins or k.numel() != bins:
        raise ValueError("null_a, null_b must be [nperm, bins, K] and dist, k [bins]")
    _lib.call("epi_null_exceedances", _ptr(null_a), _ptr(null_b), int(nperm), bins, K, _ptr(dist), _ptr(k), _stream())
    return k


def permutation_exceedances_s1(cnt_a, cnt_b, size_a, size_b, seed, perm_offset, nperm, width, bin_offset, exp1, width_a,
                               width_b, dist, k):
    """Fused S1 permutation counts: k[b] += #{p : |null(b, p)| >= |dist[b]|} over permutations perm_offset ..
    perm_offset + nperm - 1, A' scored at width_a and B' at width_b against exp1.  k: int32 [bins] (uint32 counts)."""
    _require_cuda(cnt_a, torch.int16, "cnt_a")
    _require_cuda(cnt_b, torch.int16, "cnt_b")
    _require_cuda(exp1, torch.float32, "exp1")
    _require_cuda(dist, torch.float32, "dist")
    _require_cuda(k, torch.int32, "k")
    bins, K = cnt_a.shape
    if dist.numel() != bins or k.numel() != bins or exp1.numel() != K:
        raise ValueError("dist and k must have one entry per bin, exp1 one per state")
    _lib.call("epi_permutation_exceedances_s1", _ptr(cnt_a), _ptr(cnt_b), bins, K, int(width), int(size_a), int(size_b),
              _seed(seed), int(bin_offset), int(perm_offset), int(nperm), _ptr(exp1), int(width_a), int(width_b),
              _ptr(dist), _ptr(k), _stream())
    return k


def _group_sizes(sizes):
    arr = (ctypes.c_int32 * len(sizes))(*[int(n) for n in sizes])
    return arr, ctypes.cast(arr, ctypes.c_void_p)


def _group_blocks(cnt):
    """(groups, bins, K, group stride) of a CUDA int16 [G, bins, K] tensor whose [bins, K] blocks are contiguous; the
    blocks may be spaced further apart (a bin range of a larger [G, rows, K] tensor)."""
    if not (isinstance(cnt, torch.Tensor) and cnt.is_cuda and cnt.dtype == torch.int16 and cnt.dim() == 3):
        raise TypeError("cnt must be a CUDA int16 tensor [groups, bins, K]")
    G, bins, K = cnt.shape
    if cnt.stride(2) != 1 or (bins > 1 and cnt.stride(1) != K) or (G > 1 and cnt.stride(0) < bins * K):
        raise TypeError("cnt must hold each group's [bins, K] counts contiguously")
    return G, bins, K, cnt.stride(0) if G > 1 else bins * K


def multigroup_stat(scores, sizes):
    """Multi-group statistic of every bin: scores float32 [G, bins, K] (group g at width sizes[g]) -> (T float64 [bins],
    g* uint8 [bins], s* uint8 [bins], sign int8 [bins]), see include/epilogos_b200.h."""
    _require_cuda(scores, torch.float32, "scores")
    G, bins, K = scores.shape
    if len(sizes) != G:
        raise ValueError("one size per group")
    t = torch.empty(bins, dtype=torch.float64, device=scores.device)
    g = torch.empty(bins, dtype=torch.uint8, device=scores.device)
    s = torch.empty(bins, dtype=torch.uint8, device=scores.device)
    sign = torch.empty(bins, dtype=torch.int8, device=scores.device)
    _arr, sz = _group_sizes(sizes)
    _lib.call("epi_multigroup_stat", _ptr(scores), G, bins, K, sz, _ptr(t), _ptr(g), _ptr(s), _ptr(sign), _stream())
    return t, g, s, sign


def multigroup_shuffled_counts_range(cnt, sizes, seed, perm_offset, nperm, bin_offset=0):
    """Permutations perm_offset .. perm_offset + nperm - 1 of every bin of the groups' counts cnt [G, bins, K], drawn on
    the device: int16 [nperm, G, bins, K]."""
    G, bins, K, stride = _group_blocks(cnt)
    if len(sizes) != G:
        raise ValueError("one size per group")
    out = torch.empty((nperm, G, bins, K), dtype=torch.int16, device=cnt.device)
    _arr, sz = _group_sizes(sizes)
    _lib.call("epi_multigroup_shuffled_counts_range", _ptr(cnt), stride, G, bins, K, sz, _seed(seed), int(bin_offset),
              int(perm_offset), int(nperm), _ptr(out), _stream())
    return out


def multigroup_null_exceedances(null, sizes, t, k):
    """k[b] += #{p : T of null[p, :, b] >= t[b]}.  null: float32 scores [nperm, G, bins, K]; t float64 [bins]; k int32
    [bins] holding uint32 counts (updated in place)."""
    _require_cuda(null, torch.float32, "null")
    _require_cuda(t, torch.float64, "t")
    _require_cuda(k, torch.int32, "k")
    nperm, G, bins, K = null.shape
    if len(sizes) != G or t.numel() != bins or k.numel() != bins:
        raise ValueError("one size per group, and t, k with one entry per bin")
    _arr, sz = _group_sizes(sizes)
    _lib.call("epi_multigroup_null_exceedances", _ptr(null), G, int(nperm), bins, K, sz, _ptr(t), _ptr(k), _stream())
    return k


def multigroup_s1_fused_fits(sizes, num_states):
    """Whether epi_multigroup_exceedances_s1 takes these group widths (value tables and sampler in shared memory)."""
    arr, sz = _group_sizes(sizes)
    return _lib.load().epi_multigroup_s1_fused_fits(len(sizes), int(num_states), sz) == 1


def multigroup_exceedances_s1(cnt, sizes, seed, perm_offset, nperm, bin_offset, exp1, t, k):
    """Fused S1 multi-group permutation counts: k[b] += #{p : T_null(b, p) >= t[b]} over permutations perm_offset ..
    perm_offset + nperm - 1, group g scored at width sizes[g] against exp1.  cnt int16 [G, bins, K]; k int32 [bins]."""
    G, bins, K, stride = _group_blocks(cnt)
    _require_cuda(exp1, torch.float32, "exp1")
    _require_cuda(t, torch.float64, "t")
    _require_cuda(k, torch.int32, "k")
    if len(sizes) != G or t.numel() != bins or k.numel() != bins or exp1.numel() != K:
        raise ValueError("one size per group, t and k with one entry per bin, exp1 one per state")
    _arr, sz = _group_sizes(sizes)
    _lib.call("epi_multigroup_exceedances_s1", _ptr(cnt), stride, G, bins, K, sz, _seed(seed), int(bin_offset),
              int(perm_offset), int(nperm), _ptr(exp1), _ptr(t), _ptr(k), _stream())
    return k


def _strata_sizes(sizes, groups=None):
    """(H, G, ctypes array) of the sizes [H][G] (a sequence of per-stratum group sizes)."""
    rows = [[int(v) for v in r] for r in sizes]
    G = len(rows[0]) if rows else 0
    if any(len(r) != G for r in rows) or (groups is not None and G != groups):
        raise ValueError("the strata sizes must be [strata][groups]%s" % ("" if groups is None else " with %d groups" % groups))
    flat = [v for r in rows for v in r]
    arr = (ctypes.c_int32 * max(len(flat), 1))(*flat)
    return len(rows), G, arr


def stratified_shuffled_counts_range(cnt, sizes, seed, perm_offset, nperm, bin_offset=0):
    """Permutations perm_offset .. perm_offset + nperm - 1 of every bin shuffled within strata: cnt int16 [H, bins, K]
    holds each stratum's counts over the row being shuffled (blocks may be spaced further apart), sizes [H][G] the groups'
    biosamples in each stratum.  Returns int16 [nperm, G, bins, K], the groups' counts summed over the strata."""
    H, bins, K, stride = _group_blocks(cnt)
    h, G, arr = _strata_sizes(sizes)
    if h != H:
        raise ValueError("one row of sizes per stratum")
    out = torch.empty((nperm, G, bins, K), dtype=torch.int16, device=cnt.device)
    _lib.call("epi_stratified_shuffled_counts_range", _ptr(cnt), stride, H, bins, K, ctypes.cast(arr, ctypes.c_void_p), G,
              _seed(seed), int(bin_offset), int(perm_offset), int(nperm), _ptr(out), _stream())
    return out


def stratified_exceedances_s1(cnt, sizes, cnt_a, cnt_b, seed, perm_offset, nperm, bin_offset, exp1, width_a, width_b,
                              dist, k):
    """Fused stratified S1 permutation counts of a paired comparison: k[b] += #{p : |null(b, p)| >= |dist[b]|} over
    permutations perm_offset .. perm_offset + nperm - 1 drawn as stratified_shuffled_counts_range draws them (sizes
    [H][2]), A' scored at width_a and B' = cnt_a + cnt_b - A' at width_b against exp1.  k: int32 [bins] (uint32 counts)."""
    H, bins, K, stride = _group_blocks(cnt)
    h, _, arr = _strata_sizes(sizes, groups=2)
    for t, name in ((cnt_a, "cnt_a"), (cnt_b, "cnt_b")):
        _require_cuda(t, torch.int16, name)
    _require_cuda(exp1, torch.float32, "exp1")
    _require_cuda(dist, torch.float32, "dist")
    _require_cuda(k, torch.int32, "k")
    if h != H or tuple(cnt_a.shape) != (bins, K) or tuple(cnt_b.shape) != (bins, K):
        raise ValueError("one row of sizes per stratum, and cnt_a, cnt_b [bins, K]")
    if dist.numel() != bins or k.numel() != bins or exp1.numel() != K:
        raise ValueError("dist and k must have one entry per bin, exp1 one per state")
    _lib.call("epi_stratified_exceedances_s1", _ptr(cnt), stride, H, ctypes.cast(arr, ctypes.c_void_p), _ptr(cnt_a),
              _ptr(cnt_b), bins, K, _seed(seed), int(bin_offset), int(perm_offset), int(nperm), _ptr(exp1), int(width_a),
              int(width_b), _ptr(dist), _ptr(k), _stream())
    return k


def split_counts(x, cols, num_states, members, groups):
    """Counts of the groups of column splits of x (CUDA int8 [bins, pitch]).  members: CUDA int64 [nsplit, groups - 1,
    ceil(cols / 64)] column bitsets (uint64 bit patterns), the last group of a split being the complement.  Returns an int16
    view [nsplit, groups, bins, K] holding uint16 counts whose [bins, K] blocks are contiguous and start on 16 bytes."""
    _require_cuda(x, torch.int8, "x")
    _require_cuda(members, torch.int64, "members")
    bins, pitch = x.shape
    words = (int(cols) + 63) // 64
    if members.dim() != 3 or members.shape[1] != groups - 1 or members.shape[2] != words:
        raise ValueError("members must be [nsplit, groups - 1, %d] column bitsets" % words)
    nsplit = members.shape[0]
    stride = (bins * num_states + 7) & ~7
    buf = torch.empty(max(nsplit * groups * stride, 1), dtype=torch.int16, device=x.device)
    _lib.call("epi_split_counts", _ptr(x), bins, int(cols), pitch, int(num_states), _ptr(members), nsplit, int(groups),
              _ptr(buf), _stream())
    return buf.as_strided((nsplit, groups, bins, num_states), (groups * stride, stride, num_states, 1))


def window_max(stat, window, max_inout):
    """max_inout[p] = max(max_inout[p], largest sum of `window` consecutive q(stat[p, i]) = rint(stat[p, i] * 2^24)).
    stat: CUDA float32 or float64 [nrows, n] whose rows are contiguous; max_inout: CUDA int64 [nrows], updated in place."""
    if not (isinstance(stat, torch.Tensor) and stat.is_cuda and stat.dtype in (torch.float32, torch.float64)
            and stat.dim() == 2 and (stat.shape[1] <= 1 or stat.stride(1) == 1)):
        raise TypeError("stat must be a CUDA float32 or float64 [nrows, n] tensor with contiguous rows")
    _require_cuda(max_inout, torch.int64, "max_inout")
    nrows, n = stat.shape
    if max_inout.numel() != nrows:
        raise ValueError("max_inout must have one entry per row")
    _lib.call("epi_window_max", _ptr(stat), 0 if stat.dtype == torch.float32 else 1, nrows, stat.stride(0), n,
              int(window), _ptr(max_inout), _stream())
    return max_inout


def pairwise_combine(score_a=None, score_b=None, null_a=None, null_b=None):
    """(delta float32 [rows, K] or None, null_dist float32 [rows] or None)."""
    ref = score_a if score_a is not None else null_a
    rows, k = ref.shape
    delta = torch.empty((rows, k), dtype=torch.float32, device=ref.device) if score_a is not None else None
    dist = torch.empty(rows, dtype=torch.float32, device=ref.device) if null_a is not None else None
    _lib.call("epi_pairwise_combine", _ptr(score_a), _ptr(score_b), _ptr(null_a), _ptr(null_b), rows, k, _ptr(delta),
              _ptr(dist), _stream())
    return delta, dist


def quiescent_mask(cnt_a, cols_a, cnt_b, cols_b, quiescent_state):
    _require_cuda(cnt_a, torch.int16, "cnt_a")
    _require_cuda(cnt_b, torch.int16, "cnt_b")
    bins, k = cnt_a.shape
    mask = torch.empty(bins, dtype=torch.uint8, device=cnt_a.device)
    _lib.call("epi_quiescent_mask", _ptr(cnt_a), _ptr(cnt_b), bins, k, int(cols_a), int(cols_b), int(quiescent_state),
              _ptr(mask), _stream())
    return mask


def pairwise_real_reduce(delta, text_round_trip=True):
    """(signed squared distance float32 [rows], max-difference state int32 [rows]) of the real deltas as the
    reference's paired ROI stage computes them after re-reading the 5-decimal text (roiAndVisualPairwise.py:339-354)."""
    _require_cuda(delta, torch.float32, "delta")
    rows, k = delta.shape
    dist = torch.empty(rows, dtype=torch.float32, device=delta.device)
    md = torch.empty(rows, dtype=torch.int32, device=delta.device)
    _lib.call("epi_pairwise_real_reduce", _ptr(delta), rows, k, 1 if text_round_trip else 0, _ptr(dist), _ptr(md),
              _stream())
    return dist, md


# ------------------------------------------------------------------------------------------------ paired statistics
def null_compact(null_dist, quiescent=None):
    """Null distances float32 [bins] or [nperm, bins] -> the pool float32 [nperm * count] of the bins whose quiescent flag
    (uint8 [bins]) is 0, permutation-major, bins in their order."""
    _require_cuda(null_dist, torch.float32, "null_dist")
    if quiescent is not None:
        _require_cuda(quiescent, torch.uint8, "quiescent")
    nperm, bins = (1, null_dist.shape[0]) if null_dist.dim() == 1 else tuple(null_dist.shape)
    nbytes = ctypes.c_int64(0)
    _lib.call("epi_null_compact_workspace_size", bins, ctypes.byref(nbytes))
    ws = torch.empty(max(nbytes.value, 1), dtype=torch.uint8, device=null_dist.device)
    pool = torch.empty(nperm * bins, dtype=torch.float32, device=null_dist.device)
    count = torch.zeros(1, dtype=torch.int64, device=null_dist.device)
    _lib.call("epi_null_compact", _ptr(null_dist), _ptr(quiescent), bins, nperm, _ptr(pool), _ptr(count), _ptr(ws),
              nbytes.value, _stream())
    return pool[: nperm * int(count.item())]


def null_subsample(pool, trials, size, seed):
    """(indices int32 [trials, size], samples float32 [trials, size]): trial t's keyed permutation of the pool."""
    _require_cuda(pool, torch.float32, "pool")
    idx = torch.empty((trials, size), dtype=torch.int32, device=pool.device)
    samples = torch.empty((trials, size), dtype=torch.float32, device=pool.device)
    _lib.call("epi_null_subsample", _ptr(pool), pool.numel(), int(trials), int(size), _seed(seed), _ptr(idx),
              _ptr(samples), _stream())
    return idx, samples


def gennorm_fit(samples):
    """scipy.stats.gennorm.fit of every row of samples (float32 [trials, size]) -> (params float64 [trials, 4] = beta,
    loc, scale, NLL; status int32 [trials, 2] = iterations, converged)."""
    _require_cuda(samples, torch.float32, "samples")
    trials, size = samples.shape
    params = torch.empty((trials, 4), dtype=torch.float64, device=samples.device)
    status = torch.empty((trials, 2), dtype=torch.int32, device=samples.device)
    _lib.call("epi_gennorm_fit", _ptr(samples), int(trials), int(size), _ptr(params), _ptr(status), _stream())
    return params, status


def gennorm_pvalues(x, beta, loc, scale):
    """Two-sided gennorm p-values float64 of the float32 values x."""
    _require_cuda(x, torch.float32, "x")
    p = torch.empty(x.shape, dtype=torch.float64, device=x.device)
    _lib.call("epi_gennorm_pvalues", _ptr(x), x.numel(), float(beta), float(loc), float(scale), _ptr(p), _stream())
    return p


def bh_adjust(p):
    """Benjamini-Hochberg adjusted p-values (statsmodels fdr_bh) of float64 p >= 0, in input order."""
    _require_cuda(p, torch.float64, "p")
    nbytes = ctypes.c_int64(0)
    _lib.call("epi_bh_workspace_size", p.numel(), ctypes.byref(nbytes))
    ws = torch.empty(max(nbytes.value, 1), dtype=torch.uint8, device=p.device)
    q = torch.empty_like(p)
    _lib.call("epi_bh_adjust", _ptr(p), p.numel(), _ptr(q), _ptr(ws), nbytes.value, _stream())
    return q
