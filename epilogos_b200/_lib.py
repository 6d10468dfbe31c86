"""ctypes binding of include/epilogos_b200.h (the C-ABI drop-in boundary).

The library is loaded from the package directory (built in-tree by epilogos_b200/build.py).  There is no
CPU fallback anywhere in this package: if the library is missing, or a compute entry point is called
without a B200, the call raises.
"""
import ctypes
from ctypes import c_char_p, c_double, c_int, c_int32, c_int64, c_uint64, c_void_p, POINTER
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "libepilogos_b200.so"

EPI_SCORE_TABLE = 0
EPI_SCORE_DIRECT = 1
EPI_MAX_STATES = 32
EPI_MAX_GROUPS = 64
EPI_MAX_STRATA = 64

# name -> (restype, argtypes); mirrors include/epilogos_b200.h one to one
PROTOTYPES = {
    "epi_abi_version": (c_int, []),
    "epi_last_error": (c_char_p, []),
    "epi_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "epi_bin_counts": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_void_p]),
    "epi_group_counts": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_void_p, c_int32, c_void_p,
                                 c_void_p]),
    "epi_gather_columns": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_void_p, c_int32, c_void_p, c_int64, c_void_p]),
    "epi_expected_s1s2": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "epi_normalize_i64": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "epi_scores_s1": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "epi_scores_s2": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_int32,
                              c_void_p]),
    "epi_scores_s2_fixed_point": (c_int, [c_void_p, c_int32, c_int64, c_void_p, POINTER(c_int32), c_void_p]),
    "epi_s3_plan": (c_int, [c_int64, c_int32, c_int32, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64),
                            POINTER(c_int64), POINTER(c_int64)]),
    "epi_s3_onehot": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_int64, c_int64, c_void_p]),
    "epi_s3_gram": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int32, c_void_p]),
    "epi_s3_finalize": (c_int, [c_void_p, c_int32, c_int32, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "epi_s3_terms_size": (c_int, [c_int32, c_int32, POINTER(c_int64)]),
    "epi_s3_terms": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "epi_scores_s3": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "epi_shuffled_counts_perm": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int32, c_void_p, c_int64,
                                         c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "epi_shuffled_counts_philox": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_uint64,
                                           c_int64, c_int32, c_void_p, c_void_p, c_void_p]),
    "epi_shuffled_counts_philox_range": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32,
                                                 c_uint64, c_int64, c_int64, c_int32, c_void_p, c_void_p, c_void_p]),
    "epi_null_exceedances": (c_int, [c_void_p, c_void_p, c_int32, c_int64, c_int32, c_void_p, c_void_p, c_void_p]),
    "epi_permutation_exceedances_s1": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_uint64,
                                               c_int64, c_int64, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_void_p,
                                               c_void_p]),
    "epi_multigroup_stat": (c_int, [c_void_p, c_int32, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "epi_multigroup_shuffled_counts_range": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_uint64,
                                                     c_int64, c_int64, c_int32, c_void_p, c_void_p]),
    "epi_multigroup_null_exceedances": (c_int, [c_void_p, c_int32, c_int32, c_int64, c_int32, c_void_p, c_void_p,
                                                c_void_p, c_void_p]),
    "epi_multigroup_exceedances_s1": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_uint64, c_int64,
                                              c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "epi_multigroup_s1_fused_fits": (c_int, [c_int32, c_int32, c_void_p]),
    "epi_stratified_shuffled_counts_range": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_int32,
                                                     c_uint64, c_int64, c_int64, c_int32, c_void_p, c_void_p]),
    "epi_stratified_exceedances_s1": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                                              c_uint64, c_int64, c_int64, c_int32, c_void_p, c_int32, c_int32, c_void_p,
                                              c_void_p, c_void_p]),
    "epi_split_counts": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_int32, c_int32, c_void_p,
                                 c_void_p]),
    "epi_window_max": (c_int, [c_void_p, c_int32, c_int64, c_int64, c_int64, c_int32, c_void_p, c_void_p]),
    "epi_write_permutations_gz": (c_int, [c_char_p, c_char_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_int64, c_int32, c_int32]),
    "epi_write_multigroup_gz": (c_int, [c_char_p, c_char_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_char_p, c_int32, c_char_p, c_int32, c_void_p, c_void_p, c_void_p,
                                        c_int64, c_int32, c_int32]),
    "epi_pairwise_combine": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p,
                                     c_void_p]),
    "epi_quiescent_mask": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                   c_void_p]),
    "epi_simsearch_row_norms": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_void_p]),
    "epi_simsearch_distances": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "epi_simsearch_mode_sorted": (c_int, [c_void_p, c_int32, c_int64, c_void_p, c_void_p, c_void_p]),
    "epi_simsearch_pick": (c_int, [c_void_p, c_void_p, c_int32, c_int64, c_void_p, c_void_p, c_int32, c_int32, c_void_p,
                                   c_void_p]),
    "epi_tsv_shape": (c_int, [c_char_p, POINTER(c_int64), POINTER(c_int32)]),
    "epi_tsv_parse_open": (c_int, [c_char_p, c_int32, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int32),
                                   POINTER(c_int32), POINTER(c_int32)]),
    "epi_tsv_parse_fetch": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_char_p,
                                    c_int32]),
    "epi_tsv_parse_close": (c_int, [c_void_p]),
    "epi_inflate_file": (c_int, [c_char_p, c_void_p, c_int64, POINTER(c_int64)]),
    "epi_reader_stats": (c_int, [POINTER(c_int64)]),
    "epi_reader_concurrency": (c_int, [c_int32, c_int32]),
    "epi_reader_threads": (c_int, [POINTER(c_int32), POINTER(c_int32)]),
    "epi_statebyline_read": (c_int, [c_char_p, c_void_p, c_int64, c_int64, c_int32, POINTER(c_int64), c_char_p, c_int32]),
    "epi_columns_to_rows": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_void_p, c_int64, c_int32]),
    "epi_write_matrix_tsv": (c_int, [c_char_p, c_char_p, c_void_p, c_int64, c_int32, c_int64, c_int64, c_int64, c_int32,
                                     c_int32]),
    "epi_scores_tsv_open": (c_int, [c_char_p, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int32), POINTER(c_int32),
                                    POINTER(c_int32)]),
    "epi_scores_tsv_fetch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_char_p, c_int32]),
    "epi_scores_tsv_close": (c_int, [c_void_p]),
    "epi_pack_tsv": (c_int, [c_char_p, c_int64, c_int64, c_int32, c_int32, c_void_p, c_int64, c_void_p, c_void_p,
                             c_void_p, c_void_p, c_int32, POINTER(c_int32)]),
    "epi_write_scores_gz": (c_int, [c_char_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                                    c_int32, c_int32]),
    "epi_roi_maxmean": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, POINTER(c_int32)]),
    "epi_pairwise_real_reduce": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "epi_null_compact_workspace_size": (c_int, [c_int64, POINTER(c_int64)]),
    "epi_null_compact": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "epi_null_subsample": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_uint64, c_void_p, c_void_p, c_void_p]),
    "epi_gennorm_fit": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "epi_gennorm_pvalues": (c_int, [c_void_p, c_int64, c_double, c_double, c_double, c_void_p, c_void_p]),
    "epi_bh_workspace_size": (c_int, [c_int64, POINTER(c_int64)]),
    "epi_bh_adjust": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p]),
    "epi_write_metrics_gz": (c_int, [c_char_p, c_char_p, c_void_p, c_void_p, c_void_p, c_char_p, c_int32, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32]),
    "epi_single_host": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "epi_packed_bits": (c_int, [c_int32]),
    "epi_packed_pitch": (c_int64, [c_int32, c_int32]),
    "epi_pack_states_host": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_int64, c_int32]),
    "epi_pack_states": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_int64, c_void_p]),
    "epi_unpack_states": (c_int, [c_void_p, c_int64, c_int32, c_int32, c_int64, c_void_p, c_int64, c_void_p]),
    "epi_single_host_packed": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                       c_void_p]),
    "epi_s3_host": (c_int, [c_void_p, c_int64, c_int32, c_int64, c_int32, c_void_p, c_void_p]),
    "epi_paired_host": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int32, c_int64, c_int32, c_int32, c_int32,
                                c_int32, c_uint64, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
}

_lib = None


class EpilogosB200Error(RuntimeError):
    pass


def load():
    """dlopen the library and attach prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise EpilogosB200Error(
            "%s not found: build it with `python -m epilogos_b200.build` (there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def call(name, *args):
    """Call an int-returning entry point and raise EpilogosB200Error with epi_last_error() on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.epi_last_error()
        raise EpilogosB200Error("%s failed (rc=%d): %s" % (name, rc, msg.decode() if msg else "?"))
    return rc
