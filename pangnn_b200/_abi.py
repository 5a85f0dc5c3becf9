"""ctypes binding of ``include/pangnn_b200.h`` — the only way Python reaches the CUDA kernels.

There is deliberately NO fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes as C
import os

from . import build as _build

_c_p = C.c_void_p
_i64, _i32, _sz, _f32, _f64, _int = C.c_int64, C.c_int32, C.c_size_t, C.c_float, C.c_double, C.c_int

# name -> (restype, argtypes)   — order and meaning exactly as in include/pangnn_b200.h
SIGNATURES = {
    "pangnn_abi_version": (_int, []),
    "pangnn_last_error": (C.c_char_p, []),
    "pangnn_source_digest": (C.c_char_p, []),
    "pangnn_sort_pairs_workspace_bytes": (_sz, [_i64]),
    "pangnn_sort_pairs_u64": (_int, [_c_p, _c_p, _c_p, _c_p, _i64, _int, _c_p, _sz, _c_p]),
    "pangnn_scan_workspace_bytes": (_sz, [_i64]),
    "pangnn_exclusive_scan_u32": (_int, [_c_p, _c_p, _i64, _c_p, _c_p, _sz, _c_p]),
    "pangnn_csr_build_workspace_bytes": (_sz, [_i64]),
    "pangnn_csr_build": (_int, [_c_p, _i64, _i32, _int, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_gcn_norm": (_int, [_c_p, _c_p, _c_p, _c_p, _i32, _c_p, _c_p, _c_p]),
    "pangnn_gcn_norm_apply": (_int, [_c_p, _c_p, _c_p, _c_p, _c_p, _i32, _int, _c_p, _c_p]),
    "pangnn_gcn_aggregate": (_int, [_c_p, _c_p, _c_p, _c_p, _i64, _i32, _i32, _c_p, _int, _c_p, _i64, _c_p]),
    "pangnn_act_bwd_bias": (_int, [_c_p, _c_p, _i64, _i32, _int, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_act_bwd_bias_workspace_bytes": (_sz, [_i64, _i32]),
    "pangnn_gemm_tn_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "pangnn_gemm_tn": (_int, [_c_p, _i64, _c_p, _i64, _i64, _i32, _i32, _c_p, _c_p, _sz, _c_p]),
    "pangnn_node_linear": (_int, [_c_p, _i64, _i64, _i32, _c_p, _i64, _int, _i32, _c_p, _int, _c_p, _i64, _c_p]),
    "pangnn_node_linear_push": (_int, [_c_p, _i64, _i64, _i32, _c_p, _i64, _int, _i32, _c_p, _int, _c_p, _i64,
                                       _c_p, _c_p, _i64, _i64, _c_p, _c_p, _i64, _i64, _c_p]),
    "pangnn_hits_sort_unique_workspace_bytes": (_sz, [_i64]),
    "pangnn_hits_sort_unique": (_int, [_c_p, _c_p, _c_p, _i64, _i32, _c_p, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_hits_normalize_workspace_bytes": (_sz, [_i64]),
    "pangnn_hits_normalize": (_int, [_c_p, _c_p, _c_p, _i64, _c_p, _c_p, _f64, _f64, _f64, _int,
                                     _c_p, _c_p, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_rows_gather_copy": (_int, [_c_p, _i64, _c_p, _i64, _i32, _c_p, _i64, _c_p]),
    "pangnn_rows_scatter_add": (_int, [_c_p, _i64, _c_p, _i64, _i32, _c_p, _i64, _c_p]),
    "pangnn_grad_bucket_floats": (_i64, [_c_p, _i32]),
    "pangnn_grad_push": (_int, [_c_p, _c_p, _i32, _c_p, _i64, _c_p, _i32, _i32, _c_p, _c_p]),
    "pangnn_grad_reduce": (_int, [_c_p, _c_p, _i32, _c_p, _i64, _c_p, _i32, _i32, _c_p, _i64, _c_p]),
    "pangnn_edges_sorted": (_int, [_c_p, _i64, _i32, _c_p, _c_p]),
    "pangnn_csr_from_sorted": (_int, [_c_p, _i64, _i32, _c_p, _c_p, _c_p, _c_p]),
    "pangnn_csr_transpose": (_int, [_c_p, _c_p, _c_p, _i64, _i32, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_csr_merge_band": (_int, [_c_p, _c_p, _c_p, _i64, _i64, _i32, _int, _c_p, _c_p, _c_p, _c_p]),
    "pangnn_csr_spmv2": (_int, [_c_p, _c_p, _c_p, _c_p, _i32, _c_p, _c_p, _c_p]),
    "pangnn_rank1_affine_act": (_int, [_c_p, _c_p, _c_p, _c_p, _c_p, _i64, _i32, _int, _c_p, _i64, _c_p]),
    "pangnn_rank1_bwd_workspace_bytes": (_sz, [_i64, _i32]),
    "pangnn_rank1_bwd": (_int, [_c_p, _c_p, _c_p, _c_p, _i64, _i32, _int, _c_p, _c_p, _sz, _c_p]),
    "pangnn_parse_hits_tsv_workspace_bytes": (_sz, [_i64]),
    "pangnn_tsv_line_index": (_int, [_c_p, _i64, _c_p, _i64, _c_p, _c_p, _sz, _c_p]),
    "pangnn_tsv_parse_hits": (_int, [_c_p, _i64, _c_p, _i64, _i64, _i32, _c_p, _c_p, _i32, _c_p, _c_p, _c_p, _c_p]),
    "pangnn_components_init": (_int, [_c_p, _i32, _c_p]),
    "pangnn_components_round": (_int, [_c_p, _c_p, _c_p, _i64, _c_p, _i32, _c_p, _c_p]),
    "pangnn_collate": (_int, [_c_p, _i32, _i32, _c_p, _i32, _c_p, _c_p]),
    "pangnn_neighbour_band_edges": (_i64, [_i64, _i32]),
    "pangnn_neighbour_band": (_int, [_i64, _i32, _c_p, _c_p, _c_p]),
    "pangnn_segment_max_labels_workspace_bytes": (_sz, [_i64]),
    "pangnn_segment_max_labels": (_int, [_c_p, _c_p, _c_p, _int, _i64, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_edge_score_workspace_bytes": (_sz, [_i64]),
    "pangnn_edge_score_fwd": (_int, [_c_p] * 10 + [_i64, _c_p, _f32, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_edge_score_bwd": (_int, [_c_p] * 10 + [_i64, _c_p, _c_p, _f32, _f32, _c_p, _c_p, _c_p,
                                                   _c_p, _c_p, _sz, _c_p]),
    "pangnn_edge_score_predict": (_int, [_c_p] * 10 + [_i64, _f32, _c_p, _c_p, _c_p, _c_p]),
    "pangnn_edge_split": (_int, [_c_p, _c_p, _i64, C.c_uint64, C.c_uint32, C.c_uint32, _c_p, _c_p]),
    "pangnn_edge_pair_score": (_int, [_c_p, _i64, _i32, _c_p, _c_p, _i64, _int, _c_p, _c_p]),
    "pangnn_edge_pair_score_bwd_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "pangnn_edge_pair_score_bwd": (_int, [_c_p, _i64, _i32, _i32, _i64, _c_p, _c_p, _c_p, _c_p, _c_p, _c_p,
                                          _c_p, _c_p, _int, _c_p, _c_p, _sz, _c_p]),
    "pangnn_gff_parse_lines": (_int, [_c_p, _i64, _c_p, _i64, _i64, _c_p, _i32, _c_p, _c_p, _c_p, _c_p, _c_p]),
    "pangnn_tsv_lookup_columns": (_int, [_c_p, _i64, _c_p, _i64, _i64, _c_p, _i32, _i32, _c_p, _c_p, _i32, _c_p, _c_p, _c_p]),
    "pangnn_simulate_neg_counts": (_int, [C.c_uint64, _i32, _i64, _i32, _i32, _c_p, _c_p]),
    "pangnn_simulate_edges": (_int, [C.c_uint64, _i32, _i32, _i32, _i32, _f64, _f64, _f64, _i32, _i32, _c_p, _c_p, _c_p,
                                     _i64, _i64, _c_p, _i32, _c_p, _c_p, _c_p, _c_p]),
    "pangnn_metric_runs_workspace_bytes": (_sz, [_i64]),
    "pangnn_metric_runs": (_int, [_c_p, _c_p, _int, _c_p, _i64, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_metric_reduce_workspace_bytes": (_sz, [_i64]),
    "pangnn_metric_reduce": (_int, [_c_p, _i64, _c_p, _c_p, _c_p, _sz, _c_p]),
    "pangnn_metric_curve_workspace_bytes": (_sz, [_i64]),
    "pangnn_metric_curve": (_int, [_c_p, _i64, _c_p, _c_p, _int, _c_p, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
}

ABI_VERSION = 4
_lib = None


class PangnnError(RuntimeError):
    pass


def lib_path():
    # PANGNN_B200_LIB: development override (the profiling variant of tools/scorer_phases.py)
    return os.environ.get("PANGNN_B200_LIB") or _build.LIB_PATH


def load():
    """Load (once) ``pangnn_b200/_lib/libpangnn_b200.so``.  Raises if it is absent: build it with
    ``python -m pangnn_b200.build`` (or ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise PangnnError(f"{path} is missing: the CUDA extension has not been built "
                          f"(run `python -m pangnn_b200.build`). There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    if path == _build.LIB_PATH and _build.have_sources() and lib.pangnn_source_digest().decode() != _build._digest():
        # a library older than its sources would be called with the wrong argument lists
        raise PangnnError(f"{path} is stale (csrc/ or include/ changed since it was built): "
                          f"run `python -m pangnn_b200.build`")
    if lib.pangnn_abi_version() != ABI_VERSION:
        raise PangnnError("libpangnn_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().pangnn_last_error().decode(errors="replace")
        raise PangnnError(f"{what} failed (code {rc}): {msg}")
