"""ctypes binding of the C-ABI library (include/splitp_b200.h).

The product path has no CPU fallback: if `libsplitp_b200.so` is missing or a symbol is absent this
module raises at import time.  Build with `python splitp_b200/build.py`.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsplitp_b200.so")

SPB_MAX_TAXA = 64
SPB_MAX_BATCH = 64
SPB_VAL_U32, SPB_VAL_F64 = 0, 1
SPB_S0_ROWMAJOR, SPB_S0_TILED, SPB_S0_K4MAJOR = 0, 1, 2
SPB_U8_NO_MEMSET = 1
EMPTY_KEY = 0xFFFFFFFFFFFFFFFF


class SpbSplit(C.Structure):
    _fields_ = [("n", C.c_int32), ("a", C.c_int32), ("b", C.c_int32),
                ("idx_a", C.c_uint8 * SPB_MAX_TAXA), ("idx_b", C.c_uint8 * SPB_MAX_TAXA)]


def make_split(n, idx_a, idx_b):
    """Encoded split: ordered taxon positions of both sides (order = digit significance,
    splitp/constructions.py:166-171)."""
    if n > SPB_MAX_TAXA or len(idx_a) > SPB_MAX_TAXA or len(idx_b) > SPB_MAX_TAXA:
        raise ValueError(f"at most {SPB_MAX_TAXA} taxa are supported")
    s = SpbSplit()
    s.n, s.a, s.b = n, len(idx_a), len(idx_b)
    for i, t in enumerate(idx_a):
        s.idx_a[i] = t
    for i, t in enumerate(idx_b):
        s.idx_b[i] = t
    return s


SPLIT_DTYPE = np.dtype([("n", "<i4"), ("a", "<i4"), ("b", "<i4"), ("idx_a", "u1", SPB_MAX_TAXA), ("idx_b", "u1", SPB_MAX_TAXA)])
assert SPLIT_DTYPE.itemsize == C.sizeof(SpbSplit)


def make_splits(n, sides_a, sides_b):
    """Array of encoded splits built with numpy in one go (per-split ctypes filling costs microseconds each and was
    7 % of a 2,035-split scoring step).  sides_a / sides_b: equally long sequences of position lists; all sides_a
    must have one length and all sides_b one length.  Returns (ctypes array usable as spb_split*, numpy owner)."""
    A = np.asarray(sides_a, dtype=np.int64).reshape(len(sides_a), -1)
    B = np.asarray(sides_b, dtype=np.int64).reshape(len(sides_b), -1)
    if n > SPB_MAX_TAXA or A.shape[1] > SPB_MAX_TAXA or B.shape[1] > SPB_MAX_TAXA:
        raise ValueError(f"at most {SPB_MAX_TAXA} taxa are supported")
    if A.shape[0] != B.shape[0] or (A.size and (A.min() < 0 or A.max() >= n)) or (B.size and (B.min() < 0 or B.max() >= n)):
        raise ValueError("split positions out of range")
    rec = np.zeros(A.shape[0], dtype=SPLIT_DTYPE)
    rec["n"], rec["a"], rec["b"] = n, A.shape[1], B.shape[1]
    rec["idx_a"][:, :A.shape[1]] = A
    rec["idx_b"][:, :B.shape[1]] = B
    return (SpbSplit * A.shape[0]).from_buffer(rec), rec


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: the sm_100a library has not been built (python splitp_b200/build.py). "
        "splitp_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

_p, _i, _l, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double
_sp = C.POINTER(SpbSplit)

# name -> (restype, argtypes); mirrors include/splitp_b200.h line by line
PROTOTYPES = {
    "spb_version": (_i, []),
    "spb_last_error": (C.c_char_p, []),
    "spb_launch_count": (C.c_uint64, []),
    "spb_device_info": (_i, [C.POINTER(_i)] * 3),
    "spb_sm_words": (_l, [_i, _l]),
    "spb_plane_words": (_l, [_l]),
    "spb_pack": (_i, [_p, _i, _l, _l, _i, _p, _p, _p, _p]),
    "spb_count_direct": (_i, [_p, _p, _i, _l, _l, _p, _p, _p, _p]),
    "spb_compact_tmp_words": (_l, [_l]),
    "spb_compact_direct": (_i, [_p, _p, _l, _p, _p, _p, _l, _p, _p, _p]),
    "spb_count_hash": (_i, [_p, _p, _i, _l, _l, _p, _p, _p, _l, _p, _p, _p]),
    "spb_compact_hash": (_i, [_p, _p, _p, _l, _p, _p, _p, _l, _p, _p, _p]),
    "spb_direct_merge": (_i, [_p, _p, _l, _l, _p, _p]),
    "spb_hash_merge": (_i, [_p, _p, _p, _l, _p, _p, _p, _l, _p, _p]),
    "spb_pack_wide": (_i, [_p, _i, _l, _l, _i, _p, _p, _p]),
    "spb_count_hash_wide": (_i, [_p, _p, _l, _l, _p, _p, _p, _l, _p, _p, _p, _p]),
    "spb_hash_merge_wide": (_i, [_p, _p, _p, _l, _p, _p, _p, _l, _p, _p, _p]),
    "spb_compact_hash_wide": (_i, [_p, _p, _p, _l, _p, _p, _p, _l, _p, _p]),
    "spb_thin_gram_wide": (_i, [_p, _p, _l, _p, _i, C.c_char_p, _i, _p, _p]),
    "spb_thin_filter_words": (_l, [_l]),
    "spb_thin_gram_wide_filtered": (_i, [_p, _p, _l, _p, _i, C.c_char_p, _i, _p, _l, _p, _p]),
    "spb_project_wide": (_i, [_p, _l, _i, C.c_char_p, _i, _p, _p]),
    "spb_pair_tables_wide_ws": (_l, [_l, _i]),
    "spb_pair_tables_wide": (_i, [_p, _p, _l, _i, _p, _p, _p]),
    "spb_flatten_coo": (_i, [_p, _l, _sp, _p, _p, _p]),
    "spb_flatten_dense": (_i, [_p, _p, _i, _d, _l, _sp, _p, _p]),
    "spb_flatten_dense_w": (_i, [_p, _p, _i, _d, _l, _sp, _p, _p, _p]),
    "spb_flatten_reduced_plan": (_i, [_p, _l, _sp, _p, _p, _p, C.POINTER(_l), _p]),
    "spb_flatten_reduced_fill": (_i, [_p, _p, _i, _d, _l, _sp, _p, _p, _l, _l, _p, _p]),
    "spb_flatten_reduced_fill_w": (_i, [_p, _p, _i, _d, _l, _sp, _p, _p, _l, _l, _p, _p, _p]),
    "spb_flatten_u8": (_i, [_p, _p, _l, _sp, _p, _p, _p, _l, _l, _i, _i, _p, _p, _p, _l, _p]),
    "spb_flatten_u8_clear": (_i, [_p, _l, _sp, _p, _p, _p, _l, _l, _i, _p]),
    "spb_pair_raw_words": (_l, [_i]),
    "spb_pair_tables": (_i, [_p, _p, _i, _l, _l, _l, _p, _p]),
    "spb_pair_finalize": (_i, [_p, _i, _d, _p, _p, _p, _p]),
    "spb_pair_tables_segments": (_i, [_p, _p, _i, _l, _p, _l, _p, _p]),
    "spb_pair_finalize_rows": (_i, [_p, _l, _i, _d, _p, _p, _p, _p]),
    "spb_pair_tables_weighted": (_i, [_p, _p, _l, _i, _p, _p]),
    "spb_pair_tables_count_rows": (_i, [_p, _p, _l, _l, _i, _p, _p]),
    "spb_pair_transform": (_i, [_p, _i, _p, _p, _p]),
    "spb_subflatten": (_i, [_p, _p, _i, _sp, _p, _p]),
    "spb_subflatten_score": (_i, [_p, _p, _i, _p, _p, _l, _p, _p]),
    "spb_subflatten_tables_doubles": (_l, [_i]),
    "spb_subflatten_score_tables": (_i, [_p, _p, _i, _p, _p, _l, _p, _p, _i, _p]),
    "spb_gram_f64_ws": (_l, [_l, _l, _l]),
    "spb_gram_f64": (_i, [_p, _l, _l, _l, _p, _p, _p]),
    "spb_s0_bytes": (_l, [_l, _l]),
    "spb_gram_u8_ws": (_l, [_l, _l, _i, _i]),
    "spb_gram_u8_batch": (_i, [_p, _l, _i, _l, _l, _i, _p, _l, _p, _p]),
    "spb_gram_hi_correction_batch": (_i, [_p, _l, _i, _l, _l, _i, _p, _p, _p, _l, _p, _l, _p]),
    "spb_flatten_u8_batch": (_i, [_p, _p, _l, _sp, _i, _p, _l, _l, _l, _i, _i, _p, _p, _p, _l, _p]),
    "spb_flatten_u8_clear_batch": (_i, [_p, _l, _sp, _i, _p, _l, _l, _l, _i, _p]),
    "spb_col_rank_words": (_l, [_i]),
    "spb_col_ranks_batch": (_i, [_p, _l, _sp, _i, _p, _l, _p, _p]),
    "spb_flatten_u8_batch_cols": (_i, [_p, _p, _l, _sp, _i, _p, _l, _p, _l, _l, _l, _i, _i, _p, _p, _p, _l, _p]),
    "spb_flatten_u8_clear_batch_cols": (_i, [_p, _l, _sp, _i, _p, _l, _p, _l, _l, _l, _i, _p]),
    "spb_gram_u8_batch_cols": (_i, [_p, _l, _i, _l, _l, _i, _p, _p, _l, _p, _p]),
    "spb_gram_u8": (_i, [_p, _l, _l, _i, _p, _p, _p]),
    "spb_gram_u8_simt": (_i, [_p, _l, _l, _i, _p, _p]),
    "spb_gram_hi_correction": (_i, [_p, _l, _l, _i, _p, _p, _p, _l, _p, _p]),
    "spb_score_gram_small": (_i, [_p, _l, _l, _l, _p, _p, _p]),
    "spb_score_gram_large_ws": (_l, [_l, _l]),
    "spb_score_last_unconverged": (_i, []),
    "spb_score_gram_large": (_i, [_p, _l, _l, _l, _p, _p, _p, _p]),
    "spb_score_gram_large_n": (_i, [_p, _l, _l, _l, _p, _p, _p, _i, _p]),
    "spb_gram_u8_batch_i32": (_i, [_p, _l, _i, _l, _l, _p, _l, _p]),
    "spb_gram_u8_batch_i32_cols": (_i, [_p, _l, _i, _l, _l, _p, _p, _l, _p]),
    "spb_gram_hi_strip_batch": (_i, [_p, _l, _i, _l, _l, _i, _p, _p, _p, _l, _p, _l, _p, _p, _p, _p]),
    "spb_gram_hi_strip_table_ws": (_l, [_i, _l, _l]),
    "spb_gram_hi_strip_batch_table": (_i, [_p, _p, _l, _sp, _i, _l, _l, _p, _p, _p, _l, _p, _l, _p, _p, _p, _p, _p]),
    "spb_gram_hi_strip_batch_table_cols": (_i, [_p, _p, _l, _sp, _i, _l, _l, _p, _l, _p, _p, _p, _l, _p, _l, _p, _p, _p, _p, _p]),
    "spb_score_gram_large_i32": (_i, [_p, _l, _l, _l, _p, _l, _p, _p, _p, _p, _p, _p, _p]),
    "spb_score_gram_large_i32_n": (_i, [_p, _l, _l, _l, _p, _l, _p, _p, _p, _p, _p, _p, _i, _p]),
    "spb_symv_i32_ws": (_l, [_l, _l]),
    "spb_symv_i32": (_i, [_p, _l, _l, _l, _p, _p, _p, _i, _p]),
    "spb_sparse_gram_small_ws": (_l, [_l, _l, _l]),
    "spb_sparse_gram_small": (_i, [_p, _p, _p, _p, _l, _l, _l, _p, _p, _p]),
    "spb_score_sparse_large_ws": (_l, [_l, _l, _l, _l]),
    "spb_score_sparse_large_n": (_i, [_p, _p, _p, _p, _p, _p, _l, _l, _l, _l, _p, _p, _p, _i, _p]),
    "spb_sparse_product_ws": (_l, [_l, _l, _l, _l]),
    "spb_sparse_product": (_i, [_p, _p, _p, _p, _p, _p, _l, _l, _l, _l, _p, _p, _p, _p]),
    "spb_mi_partials": (_l, []),
    "spb_marginals_dense": (_i, [_p, _l, _l, _l, _p, _p, _p]),
    "spb_mi_dense": (_i, [_p, _l, _l, _l, _p, _p, _p, _p, _p]),
    "spb_outer_f64": (_i, [_p, _l, _p, _l, _p, _i, _p]),
    "spb_flatten_coo_banned": (_i, [_p, _l, _sp, _i, _i, _p, _p, _p, _p]),
    "spb_table_marginals": (_i, [_p, _p, _i, _l, _sp, _i, _i, _p, _p, _l, _p, _p, _l, _p, _p]),
    "spb_mi_table": (_i, [_p, _p, _i, _d, _l, _sp, _p, _p, _l, _p, _p, _l, _p, _p, _p]),
    "spb_mi_side_cap": (_l, [_l, _i]),
    "spb_mi_scores_ws": (_l, [_l, _i, _l, _l]),
    "spb_mi_scores": (_i, [_p, _i, _p, _i, _d, _l, _p, _l, _l, _p, _p, _p]),
    "spb_mi_row_slots": (_i, [_p, _i, _l, _p, _l, _l, _p, _p, _p]),
    "spb_mi_rows_ws": (_l, [_l, _l, _l, _l]),
    "spb_mi_row_scores": (_i, [_p, _l, _p, _p, _l, _d, _p, _l, _l, _p, _p, _p, _p]),
    "spb_bootstrap_counts": (_i, [_p, _l, _l, C.c_uint64, _l, _l, _p, _p]),
    "spb_bootstrap_compact_ws": (_l, [_l, _l]),
    "spb_bootstrap_compact": (_i, [_p, _p, _i, _l, _l, _p, _p, _l, _p, _p, _p]),
    "spb_subflatten_score_tables_multi": (_i, [_p, _p, _i, _p, _p, _l, _l, _p, _p]),
    "spb_subflatten_score_multi": (_i, [_p, _p, _i, _p, _p, _l, _l, _p, _p]),
    "spb_quartet_tables": (_i, [_p, _p, _i, _l, _l, _l, _p, _l, _p, _p]),
    "spb_quartet_flattening_ws": (_l, [_l]),
    "spb_quartet_flattening_scores": (_i, [_p, _l, _p, _p, _p]),
    "spb_quartet_mi_scores": (_i, [_p, _l, _p, _p]),
    "spb_agglomerate_ws_bytes": (_l, [_i, _l]),
    "spb_agglomerate_init": (_i, [_i, _l, _i, _p, _p, _p, _p]),
    "spb_agglomerate_step": (_i, [_i, _l, _i, _i, _p, _p, _p, _p, _p, _p, _p]),
}

for _name, (_res, _args) in PROTOTYPES.items():
    _f = getattr(lib, _name)  # AttributeError here = the library is stale: rebuild it
    _f.restype = _res
    _f.argtypes = _args

_ERRORS = {1: ValueError, 2: RuntimeError, 3: MemoryError, 4: NotImplementedError}


def check(rc):
    """Maps an spb_status to the Python exception the reference would raise for that condition."""
    if rc != 0:
        msg = lib.spb_last_error().decode("utf-8", "replace")
        raise _ERRORS.get(rc, RuntimeError)(f"splitp_b200: {msg}")


def call(name, *args):
    check(getattr(lib, name)(*args))
