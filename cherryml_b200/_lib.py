"""ctypes binding of the C ABI declared in ``include/cherryml_b200.h``.

There is no CPU fallback: if the shared library is missing, or a call fails, this module
raises.  PyTorch is used by the callers only to own device memory and streams.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_int, c_int32, c_int64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcherryml_b200.so")

# numpy dtypes of the two descriptor structs (must match include/cherryml_b200.h)
FAM_DESC_DTYPE = np.dtype(
    [
        ("msa_off", np.int64),
        ("row_stride", np.int32),
        ("n_chunks", np.int32),
        ("aux_off", np.int32),
        ("aux_cnt", np.int32),
        ("rate_off", np.int32),
        ("n_rates", np.int32),
    ],
    align=True,
)
TILE_DTYPE = np.dtype(
    [
        ("fam", np.int32),
        ("pair_begin", np.int32),
        ("n_pairs", np.int32),
        ("reserved", np.int32),
    ],
    align=True,
)
FC_FAMILY_DTYPE = np.dtype(
    [
        ("msa_off", np.int64),
        ("n_seqs", np.int32),
        ("row_stride", np.int32),
        ("n_sites", np.int32),
        ("cherry_off", np.int32),
        ("site_off", np.int32),
        ("seq_off", np.int32),
    ],
    align=True,
)
LL_NODE_DTYPE = np.dtype(
    [("depth", np.int32), ("flags", np.int32), ("obs_row", np.int32), ("reserved", np.int32)], align=True
)
assert FAM_DESC_DTYPE.itemsize == 32 and TILE_DTYPE.itemsize == 16 and FC_FAMILY_DTYPE.itemsize == 32
assert LL_NODE_DTYPE.itemsize == 16

NO_BUCKET = 255
# The skip code of a residue byte is the number of states S itself (bytes are in [0, S]).
MAX_BUCKETS = 254


class CherryError(RuntimeError):
    pass


_P = c_void_p
_SIGNATURES = {
    "cherry_last_error": (c_char_p, []),
    "cherry_version": (c_char_p, []),
    "cherry_launch_count": (c_int64, []),
    "cherry_reset_launch_count": (None, []),
    "cherry_count_lg": (c_int, [_P, _P, _P, _P, _P, c_int, _P, _P, c_int, c_int, c_int, _P, _P]),
    "cherry_build_bucket_table_tiles": (c_int, [_P, _P, c_int, _P, _P, _P, c_int, c_int, _P, _P]),
    "cherry_sort_pairs_by_bucket": (c_int, [_P, c_int, c_int64, c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cherry_count_co": (c_int, [_P, _P, _P, c_int64, c_int, c_int, c_int, _P, _P]),
    "cherry_validate_residues": (c_int, [_P, c_int64, c_int, _P, _P]),
    "cherry_count_per_site": (c_int, [_P, _P, _P, c_int64, c_int, c_int64, _P, c_int, c_int, _P, _P]),
    "cherry_symmetrize_lg": (c_int, [_P, c_int, c_int, c_int, _P, _P]),
    "cherry_symmetrize_co": (c_int, [_P, c_int, c_int, c_int, _P, _P]),
    "cherry_fit_workspace_bytes": (c_int, [c_int, c_int, c_int, _P]),
    "cherry_fit_init": (c_int, [_P, _P]),
    "cherry_fit_run": (c_int, [_P, c_int, _P]),
    "cherry_fit_loss_grad": (c_int, [_P, _P]),
    "cherry_fit_epoch_local": (c_int, [_P, _P, _P]),
    "cherry_fit_epoch_update": (c_int, [_P, _P, _P]),
    "cherry_fit_schedule": (c_int, [_P, _P, _P, _P]),
    "cherry_fit_symmetric_form": (c_int, [_P]),
    "cherry_expm_batched": (c_int, [_P, _P, _P]),
    "cherry_gemm_f64_batched": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "cherry_gemm_desc_bytes": (ctypes.c_size_t, [c_int]),
    "cherry_ingest_lg": (c_int, [c_char_p, c_char_p, c_char_p, _P, c_int, _P, c_int, c_char_p, c_int, c_int,
                                 c_int, _P]),
    "cherry_ingest_co": (c_int, [c_char_p, c_char_p, c_char_p, _P, c_int, _P, c_int, c_char_p, c_int, c_int,
                                 c_int, c_int, _P]),
    "cherry_ingest_free": (None, [_P]),
    "cherry_tree_ll_units_per_block": (c_int, [c_int, c_int]),
    "cherry_tree_ll_scratch_bytes": (ctypes.c_size_t, [c_int, c_int, c_int, c_int]),
    "cherry_tree_ll_transpose": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "cherry_tree_log_likelihood": (c_int, [_P, c_int, _P, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P,
                                           ctypes.c_size_t, _P, _P]),
    "cherry_tree_ll_posterior_scratch_bytes": (ctypes.c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int, _P]),
    "cherry_tree_ll_posterior": (c_int, [_P, c_int, c_int, _P, c_int, _P, c_int, _P, _P, _P, c_int, c_int, _P,
                                         ctypes.c_size_t, _P, _P, _P, _P]),
    "cherry_tree_ll_edge_derivatives_scratch_bytes": (ctypes.c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int,
                                                                        _P]),
    "cherry_tree_ll_edge_derivatives": (c_int, [_P, c_int, c_int, _P, c_int, _P, c_int, _P, _P, _P, _P, c_int, c_int,
                                                _P, ctypes.c_size_t, _P, _P, _P, _P, _P]),
    "cherry_tree_ll_pair_posterior_scratch_bytes": (ctypes.c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "cherry_tree_ll_pair_posterior": (c_int, [_P, c_int, c_int, _P, _P, c_int, _P, _P, c_int, c_int, _P,
                                              ctypes.c_size_t, _P, _P, _P, _P]),
    "cherry_fc_read_msas": (c_int, [_P, c_int, _P, c_int, c_int, c_int, _P]),
    "cherry_fc_free_msas": (None, [_P]),
    "cherry_fc_write_outputs": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, _P, c_int, _P, _P, _P, _P, _P, _P, c_int]),
    "cherry_write_count_matrices": (c_int, [c_char_p, _P, c_int, _P, c_int, _P, c_int, c_int]),
    "cherry_read_count_matrices_header": (c_int, [c_char_p, _P, _P]),
    "cherry_read_count_matrices": (c_int, [c_char_p, c_int, c_int, _P, _P, _P, ctypes.c_size_t, c_int]),
    "cherry_write_labelled_matrix": (c_int, [c_char_p, _P, c_int, _P, c_int]),
    "cherry_fc_lengths_and_rates": (c_int, [_P, c_int, _P, _P, _P, c_int, _P, c_int, c_int, _P, _P, c_int]),
    "cherry_fc_count_layout": (c_int, [_P, c_int, _P, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, c_int]),
    "cherry_fc_relayout_lg": (c_int, [_P, _P, _P, c_int, _P, _P, _P, _P, _P]),
    "cherry_fc_scratch_bytes": (ctypes.c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int]),
    "cherry_fc_pair": (c_int, [_P, _P, c_int, c_int64, c_int, ctypes.c_uint32, _P, _P, _P, _P, ctypes.c_size_t, _P]),
    "cherry_fc_ble": (c_int, [_P, _P, c_int, c_int64, c_int, _P, _P, _P, c_int, c_int, _P, _P, c_int, _P, _P, _P,
                              _P, ctypes.c_size_t, _P]),
    "cherry_count_lg_host": (
        c_int,
        [_P, c_int64, _P, c_int, _P, _P, _P, c_int64, _P, c_int64, _P, c_int64, _P, c_int,
         _P, c_int, c_int, c_int, c_int, _P, _P, _P],
    ),
}

class IngestResult(ctypes.Structure):
    """``cherry_ingest_result`` of include/cherryml_b200.h."""

    _fields_ = [
        ("kind", c_int32), ("pinned", c_int32), ("msa_bytes", c_int64), ("msa", c_void_p),
        ("n_fams", c_int32), ("r_pad", c_int32), ("fams", c_void_p),
        ("n_pairs", c_int64), ("pair_a", c_void_p), ("pair_b", c_void_p), ("pair_t", c_void_p),
        ("pair_fam", c_void_p),
        ("n_rate_vals", c_int64), ("rate_vals", c_void_p),
        ("n_aux", c_int64), ("aux", c_void_p),
        ("n_tiles", c_int32), ("max_row_stride", c_int32), ("tiles", c_void_p),
        ("n_items_examined", c_int64),
    ]


class FcMsas(ctypes.Structure):
    """``cherry_fc_msas`` of include/cherryml_b200.h."""

    _fields_ = [
        ("n_fams", c_int32), ("pinned", c_int32), ("msa_bytes", c_int64), ("msa", c_void_p), ("fams", c_void_p),
        ("total_seqs", c_int64), ("total_sites", c_int64), ("total_cherries", c_int64),
        ("name_blob", c_void_p), ("name_off", c_void_p),
    ]


_lib = None


def exported_symbols():
    """Names ``include/cherryml_b200.h`` declares (kept in sync by tests/test_abi.py)."""
    return sorted(_SIGNATURES.keys())


def load():
    """Load the library (once).  Raises ``CherryError`` if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CherryError(
            f"{LIB_PATH} not found: the CUDA library has not been built. Run "
            "`python -m cherryml_b200.csrc.build` (or __graft_entry__.build()). "
            "cherryml_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().cherry_last_error().decode("utf-8", "replace")
        raise CherryError(f"{what} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(load().cherry_launch_count())


def reset_launch_count() -> None:
    load().cherry_reset_launch_count()


def ptr(t) -> int:
    """Device (or host) address of a torch tensor / numpy array; 0 for None."""
    if t is None:
        return 0
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


def current_stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
