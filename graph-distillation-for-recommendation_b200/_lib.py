"""ctypes binding of libgdr_b200.so — the C ABI declared in include/gdr.h.

This is the whole "extension": no torch types cross the boundary, only raw device
pointers (``tensor.data_ptr()``), sizes and the current CUDA stream handle.  There
is deliberately NO fallback: if the shared library is missing or a call fails the
caller gets an exception, never a CPU/eager result.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libgdr_b200.so")

i64, i32, f32, vp, cp = C.c_int64, C.c_int, C.c_float, C.c_void_p, C.c_char_p

# name -> (restype, argtypes).  Pointers are passed as integers (void*).
_SIGNATURES = {
    "gdr_abi_version": (i32, []),
    "gdr_last_error": (cp, []),
    "gdr_device_info": (i32, [vp, vp, vp]),
    "gdr_launch_count": (i64, []),
    "gdr_debug_set": (i32, [cp, i32]),
    "gdr_debug_get": (i32, [cp, vp]),
    "gdr_debug_mma_probe": (i32, [i32, i32, i32, vp]),
    "gdr_profile_enable": (i32, [i32]),
    "gdr_profile_collect": (i32, [vp, vp]),
    "gdr_sort_pairs_ws_bytes": (i64, [i64]),
    "gdr_sort_pairs": (i32, [i64, i32, vp, vp, vp, i64, vp]),
    "gdr_coo_to_csr_ws_bytes": (i64, [i64, i64, i64, i32]),
    "gdr_coo_to_csr": (i32, [i64, i64, i64, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_sym_normalize_ws_bytes": (i64, [i64, i64]),
    "gdr_sym_normalize": (i32, [i64, i64, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_sym_normalize_block_ws_bytes": (i64, [i64]),
    "gdr_sym_normalize_block_degrees": (i32, [i64, i64, vp, vp, vp, i32, vp, vp, vp, i64, vp]),
    "gdr_sym_normalize_block_fill": (i32, [i64, i64, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_sym_normalize_dense_ws_bytes": (i64, [i64]),
    "gdr_sym_normalize_dense": (i32, [i64, vp, i64, vp, i64, vp, i64, vp]),
    "gdr_bipartite_normalize": (i32, [i64, i64, i64, vp, vp, vp, vp, vp, f32, vp, vp, vp, vp, vp]),
    "gdr_csr_locate": (i32, [i64, i64, i64, vp, vp, i64, vp, vp, vp, vp, vp]),
    "gdr_lightgcn_edge_grad": (i32, [i64, i64, i64, vp, vp, vp, i32, i64, vp, vp, vp, vp, i64, f32, vp, vp, vp]),
    "gdr_bipartite_normalize_backward_ws_bytes": (i64, [i64, i64]),
    "gdr_bipartite_normalize_backward": (i32, [i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, f32, vp, vp, i64, vp, vp, vp,
                                               i64, vp]),
    "gdr_bipartite_pow_normalize": (i32, [i64, i64, i64, vp, vp, vp, vp, vp, f32, f32, vp, vp, vp, vp, vp, vp]),
    "gdr_csr_transpose_ws_bytes": (i64, [i64, i64, i64]),
    "gdr_csr_transpose": (i32, [i64, i64, i64, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_csr_to_coo": (i32, [i64, vp, vp, vp, vp, vp]),
    "gdr_spmm_prop": (i32, [i64, i64, vp, vp, vp, f32, vp, i64, vp, i64, vp, i64, f32, vp]),
    "gdr_spmm_plan_blocks": (i64, [i64, i64]),
    "gdr_spmm_plan": (i32, [i64, i64, vp, vp, vp]),
    "gdr_spmm_prop_planned": (i32, [i64, i64, vp, vp, vp, f32, vp, i64, vp, i64, vp, i64, f32, vp, i64, vp]),
    "gdr_remap_chunk_major": (i32, [i64, vp, i64, i64, i64, vp, vp]),
    "gdr_scale_rows": (i32, [i64, i64, f32, vp, i64, vp, i64, vp]),
    "gdr_center_columns_ws_bytes": (i64, [i64, i64]),
    "gdr_center_columns": (i32, [i64, i64, vp, i64, vp, vp, vp, i64, vp, i64, vp]),
    "gdr_standard_scale_ws_bytes": (i64, [i64, i64]),
    "gdr_standard_scale": (i32, [i64, i64, vp, i64, vp, i64, vp, vp, vp, i64, vp]),
    "gdr_column_sums": (i32, [i64, i64, vp, i64, vp, vp, i64, vp]),
    "gdr_center_apply": (i32, [i64, i64, vp, i64, vp, vp, i64, vp]),
    "gdr_coarse_scatter_dense": (i32, [i64, i64, vp, vp, vp, vp, vp, vp, vp]),
    "gdr_dense_to_coarse_ws_bytes": (i64, [i64]),
    "gdr_dense_to_coarse": (i32, [i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_row_sums_f32": (i32, [i64, vp, vp, vp, vp]),
    "gdr_er_lower": (i32, [i64, i64, vp, vp, vp, vp, vp, vp]),
    "gdr_edge_cosine_scale": (i32, [i64, i64, i64, vp, vp, vp, vp, i64, f32, vp, vp, vp]),
    "gdr_softmax_rows": (i32, [i64, i64, vp, i64, vp, i64, vp]),
    "gdr_class_edge_weight": (i32, [i64, i64, vp, vp, vp, vp, i64, i64, vp, vp]),
    "gdr_induced_subgraph_ws_bytes": (i64, [i64, i64]),
    "gdr_induced_subgraph_coo": (i32, [i64, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_sparsify_classes_ws_bytes": (i64, [i64, i64, i64]),
    "gdr_sparsify_classes": (i32, [i64, i64, i64, vp, vp, vp, vp, vp, i64, i64, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_topk_filter_ws_bytes": (i64, [i64, i64]),
    "gdr_topk_filter_csr": (i32, [i64, i64, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_kmeans_assign_ws_bytes": (i64, [i64, i64, i64, i32]),
    "gdr_kmeans_assign": (i32, [i64, i64, i64, vp, i64, vp, i64, vp, vp, vp, vp, i32, vp, i64, vp]),
    "gdr_kmeans_tc_xsplit_bytes": (i64, [i64, i64]),
    "gdr_kmeans_tc_prepare": (i32, [i64, i64, vp, i64, vp, i64, vp]),
    "gdr_kmeans_assign_tc_ws_bytes": (i64, [i64, i64, i64]),
    "gdr_kmeans_assign_tc": (i32, [i64, i64, i64, vp, i64, vp, vp, i64, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_kmeans_lloyd_ws_bytes": (i64, [i64, i64, i64, i32]),
    "gdr_kmeans_lloyd": (i32, [i64, i64, i64, vp, i64, vp, i64, vp, i32, C.c_double, i32, vp, vp, vp, i32, vp, i64, vp]),
    "gdr_kmeans_plusplus_ws_bytes": (i64, [i64, i64, i64, i32]),
    "gdr_kmeans_plusplus": (i32, [i64, i64, i64, vp, i64, i64, vp, i32, vp, i64, vp, vp, i64, vp]),
    "gdr_minibatch_update": (i32, [i64, i64, i64, vp, i64, vp, vp, i64, vp, i64, vp, vp]),
    "gdr_segment_sum_ws_bytes": (i64, [i64, i64, i64]),
    "gdr_segment_sum": (i32, [i64, i64, i64, vp, i64, vp, vp, i64, vp, vp, i64, vp]),
    "gdr_label_histogram": (i32, [i64, i64, vp, vp, vp, vp]),
    "gdr_kmeans_finalize": (i32, [i64, i64, vp, i64, vp, vp, i64, vp, i64, vp, i32, vp]),
    "gdr_kmeans_relocate_ws_bytes": (i64, [i64, i64, i64]),
    "gdr_kmeans_relocate": (i32, [i64, i64, i64, vp, i64, vp, i64, vp, vp, i64, vp, vp, i64, vp]),
    "gdr_inertia_ws_bytes": (i64, [i64, i64]),
    "gdr_inertia": (i32, [i64, i64, vp, i64, vp, i64, vp, vp, vp, i64, vp]),
    "gdr_add_row_vector": (i32, [i64, i64, vp, i64, vp, f32, vp]),
    "gdr_comm_unique_id": (i32, [vp]),
    "gdr_comm_init": (i32, [vp, vp, i32, i32]),
    "gdr_comm_destroy": (i32, [vp]),
    "gdr_comm_info": (i32, [vp, vp, vp, vp]),
    "gdr_allgather_rows": (i32, [vp, vp, i64, i64, vp, vp]),
    "gdr_allgather_bytes": (i32, [vp, vp, i64, vp, vp]),
    "gdr_allreduce_centroids": (i32, [vp, vp, i64, vp, i64, vp]),
    "gdr_allreduce_f64": (i32, [vp, vp, i64, i32, vp]),
    "gdr_alltoallv": (i32, [vp, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_symm_create": (i32, [vp, i64, vp]),
    "gdr_symm_destroy": (i32, [vp]),
    "gdr_symm_info": (i32, [vp, vp, vp]),
    "gdr_symm_barrier": (i32, [vp, vp]),
    "gdr_symm_put_rows": (i32, [vp, i64, vp, i64, i64, i32, vp]),
    "gdr_symm_scatterv": (i32, [vp, vp, vp, vp, vp, i64, vp]),
    "gdr_spmm_prop_mc": (i32, [vp, i64, i64, i64, i64, i64, vp, vp, vp, f32, vp, i64, vp, i64, vp, i64, f32, vp, i64, vp]),
    "gdr_kmeans_lloyd_dist": (i32, [vp, i64, i64, i64, i64, vp, i64, vp, i64, vp, i32, C.c_double, i32, vp, vp, vp, i32, vp,
                                    i64, vp]),
    "gdr_coarse_records": (i32, [i64, i64, vp, vp, vp, vp, vp, vp]),
    "gdr_coarse_merge_ws_bytes": (i64, [i64]),
    "gdr_coarse_merge": (i32, [i64, vp, i64, i64, i64, i64, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_bipartite_norm_block": (i32, [i64, i64, vp, vp, vp, vp, vp, f32, vp, vp]),
    "gdr_column_moments": (i32, [i64, i64, vp, i64, vp, vp, vp, i64, vp]),
    "gdr_standardize_apply": (i32, [i64, i64, vp, i64, vp, vp, vp, i64, vp]),
    "gdr_dense_gram_ws_bytes": (i64, [i64, i64, i64]),
    "gdr_dense_gram": (i32, [i64, i64, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp]),
    "gdr_dense_chol": (i32, [i64, vp, i64, vp, i64, vp, C.c_double, vp]),
    "gdr_dense_trsm_rows": (i32, [i64, i64, vp, i64, vp, i64, vp]),
    "gdr_dense_gemm_small": (i32, [i64, i64, i64, C.c_double, vp, i64, vp, i64, C.c_double, vp, i64, vp, i64, vp, vp]),
    "gdr_sym_eig_jacobi_ws_bytes": (i64, [i64]),
    "gdr_sym_eig_jacobi": (i32, [i64, vp, vp, vp, vp, i32, C.c_double, vp, vp, i64, vp]),
    "gdr_dense_gather_cols": (i32, [i64, i64, vp, vp, vp, vp]),
    "gdr_edges_route_ws_bytes": (i64, [i64, i32]),
    "gdr_edges_route": (i32, [i64, vp, vp, i64, i64, i32, i64, i32, vp, vp, vp, vp, i64, vp]),
    "gdr_csr_from_keys_ws_bytes": (i64, [i64]),
    "gdr_csr_from_keys": (i32, [i64, vp, i64, i64, i64, i32, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_coarsen_route_ws_bytes": (i64, [i64]),
    "gdr_coarsen_route": (i32, [i64, vp, vp, i64, vp, vp, vp, vp, vp, i64, i64, i32, i32, vp, vp, vp, vp, i64, vp]),
    "gdr_coarse_merge_edges_ws_bytes": (i64, [i64]),
    "gdr_coarse_merge_edges": (i32, [i64, vp, vp, i64, i64, i64, i64, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_cluster_stats": (i32, [i64, vp, vp, vp, i64, vp, vp, vp, vp, vp]),
    "gdr_coarse_merge_edges_dense_ok": (i32, [i64, i64, i32]),
    "gdr_coarse_merge_edges_dense_ws_bytes": (i64, [i64, i64]),
    "gdr_coarse_merge_edges_dense": (i32, [i64, vp, vp, i64, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_coarsen_ws_bytes": (i64, [i64, i64, i64]),
    "gdr_coarsen": (i32, [i64, vp, vp, i64, vp, vp, vp, vp, vp, i64, i64, i32, vp, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_coarsen_scale": (i32, [i64, vp, vp, vp, vp, vp, vp, vp]),
    "gdr_topk_scores_ws_bytes": (i64, [i64, i64, i64, i64]),
    "gdr_topk_scores": (i32, [i64, i64, i64, i64, i64, vp, i64, vp, vp, i64, vp, vp, vp, i64, vp, i64, vp, vp, i64, vp]),
    "gdr_ranking_metrics_ws_bytes": (i64, [i64, i32]),
    "gdr_ranking_metrics": (i32, [i64, i64, i64, vp, i64, vp, vp, vp, i32, vp, vp, vp, vp, vp, i64, vp]),
    "gdr_bpr_sample": (i32, [i64, i64, vp, vp, i64, vp, C.c_uint64, i64, i64, vp, vp, vp, vp]),
    "gdr_bpr_loss_ws_bytes": (i64, [i64, i64, i64]),
    "gdr_bpr_loss": (i32, [i64, i64, i64, i64, vp, i64, vp, i64, vp, vp, vp, vp, vp, i64, vp, i64, vp, vp, i64, vp]),
}

ERROR_NAMES = {-1: "GDR_EINVAL", -2: "GDR_EWORKSPACE", -3: "GDR_ECUDA", -4: "GDR_ERANGE",
               -5: "GDR_EUNSUPPORTED"}


class GdrError(RuntimeError):
    """A libgdr_b200 entry point returned a non-zero status."""

    def __init__(self, fn: str, code: int, msg: str):
        self.fn, self.code = fn, code
        super().__init__(f"{fn} -> {ERROR_NAMES.get(code, code)}: {msg}")


_lib = None


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
            "There is no CPU fallback for the distillation core."
        )
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.gdr_abi_version() != 1:
        raise ImportError("libgdr_b200.so ABI version mismatch")
    _lib = lib
    return lib


def call(name: str, *args):
    """Invoke an int-returning entry point and raise GdrError on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise GdrError(name, rc, lib.gdr_last_error().decode("utf-8", "replace"))
    return rc


def query(name: str, *args) -> int:
    """Invoke a *_ws_bytes / counter style entry point (returns its value)."""
    return int(getattr(load(), name)(*args))
