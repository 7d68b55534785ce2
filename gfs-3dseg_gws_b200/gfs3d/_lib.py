"""ctypes binding of libgfs3d.so (the C ABI declared in include/gfs3d.h).

The product path has NO fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgfs3d.so")

_i, _i64, _p, _f, _u32 = ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_float, ctypes.c_uint32

# name -> argtypes; every function returns int (gfs_status) except the three utilities
SIGNATURES = {
    "gfs_knn_f32": [_p, _i64, _i, _i, _i, _i, _p, _p, _p, _p],
    "gfs_knn_tc_f32": [_p, _i64, _i, _i, _i, _i, _p, _p, _i64, _p, _p, _p],
    "gfs_knn_tc_set_f32": [_p, _i64, _i, _i, _i, _i, _p, _p, _i64, _p, _p],
    "gfs_knn_tc_diag_f32": [_p, _i64, _i, _i, _i, _i, _p, _p, _i64, _p, _p, _p, _p],
    "gfs_pointwise_f32": [_p, _i64, _i, _i, _i, _p, _p, _i, _p, _p],
    "gfs_edge_pq_f32": [_p, _i64, _i, _i, _i, _p, _p, _p, _p, _p],
    "gfs_edgeconv_fwd": [_p, _p, _p, _p, _p, _i, _i, _i, _p, _i64, _p, _i, _i, _p, _i, _i, _p, _p],
    "gfs_pack_weight_bf16": [_p, _p, _i, _i, _p, _p],
    "gfs_cm_to_act": [_p, _i64, _i, _i, _i, _p, _i, _i, _p],
    "gfs_linear_bf16": [_p, _i, _i, _i, _p, _p, _i, _i, _i, _i, _p, _i, _i, _p, _i64, _p],
    "gfs_attention_fwd": [_p, _i, _i, _i, _i, _f, _p, _i64, _p, _i, _i, _p],
    "gfs_gw_project": [_p, _i64, _i, _i, _i, _p, _i, _i, _p, _i, _i, _p, _p, _p],
    "gfs_gw_project_tc": [_p, _i64, _i, _i, _i, _p, _i, _i, _p, _i, _i, _p, _p, _p, _i64, _p],
    "gfs_kmeans_assign_tc": [_p, _i64, _i64, _i, _i, _p, _i, _i, _p, _p, _p, _i64, _p],
    "gfs_cos_logits": [_p, _i64, _i, _i, _i, _p, _i, _i, _p, _i, _p, _f, _p, _p],
    "gfs_softmax_pool": [_p, _p, _i64, _i, _i, _i, _i, _p, _p, _p, _p],
    "gfs_refine_proto": [_p, _p, _p, _i, _i, _i, _i, _p, _p],
    "gfs_joint_histogram_i32": [_p, _p, _i64, _i, _i, _p, _p],
    "gfs_kmeans_assign": [_p, _i64, _i, _p, _i, _i, _p, _p, _p, _p],
    "gfs_kmeans_accumulate": [_p, _i64, _i, _p, _i, _p, _p, _p, _p, _p],
    "gfs_kmeans_pack": [_p, _p, _i64, _p, _i, _i, _p, _p, _p],
    "gfs_kmeans_update": [_p, _p, _i, _i, _i, _p, _p, _p, _p],
    "gfs_kmeans_pp_trial": [_p, _i64, _i64, _i, _p, _p, _i, _p, _p, _p, _p, _p],
    "gfs_kmeans_accumulate_weighted": [_p, _i64, _i, _p, _p, _i, _p, _p, _p, _p, _p],
    "gfs_kmeans_inertia": [_p, _i64, _i, _p, _p, _i, _p, _p, _p, _p],
    # training path
    "gfs_gemm_f32": [_p, _i64, _i, _i64, _p, _i64, _i, _i64, _p, _i64, _i, _i64, _p, _i, _i, _i, _i, _i, _p, _i, _p],
    "gfs_gemm_tf32": [_p, _i64, _i, _i64, _p, _i64, _i, _i64, _p, _i64, _i, _i64, _p, _i, _i, _i, _i, _i, _p, _i, _i, _p],
    "gfs_bn_stats": [_p, _i64, _i, _i64, _p, _p, _p, _p],
    "gfs_bn_act_fwd": [_p, _i64, _p, _i64, _i, _i64, _p, _p, _f, _p],
    "gfs_bn_stats_coeffs": [_p, _i64, _i, _i64, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p],
    "gfs_bn_update_running": [_p, _p, _i, _i64, _f, _p, _p, _p, _p],
    "gfs_bn_act_max_fwd": [_p, _i, _i64, _i, _p, _p, _f, _p, _i64, _p, _p],
    "gfs_bn_bwd_sums": [_p, _i64, _p, _i64, _i, _i64, _p, _p, _p, _p, _f, _p, _p, _p, _p],
    "gfs_edge_scatter_bn": [_p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _f, _p, _p, _p, _p],
    "gfs_edge_reverse_index": [_p, _i, _i, _i, _p, _p, _p],
    "gfs_edge_scatter_bn_ordered": [_p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _f, _p, _p, _p, _p, _p],
    "gfs_bn_act_bwd": [_p, _i64, _p, _i64, _p, _i64, _i, _i64, _p, _p, _p, _p, _f, _p, _p, _p, _p],
    "gfs_bn_act_bwd_argmax": [_p, _i64, _p, _i, _p, _i64, _p, _i64, _i, _i64, _p, _p, _p, _p, _f, _p, _p, _p, _p],
    "gfs_bn_act_bwd_frozen": [_p, _i64, _p, _i64, _p, _i64, _i, _i64, _p, _p, _p, _p, _f, _p, _p, _p, _p],
    "gfs_bn_act_bwd_argmax_frozen": [_p, _i64, _p, _i, _p, _i64, _p, _i64, _i, _i64, _p, _p, _p, _p, _f, _p, _p, _p, _p],
    "gfs_edge_gather": [_p, _p, _i, _i, _i, _p, _p],
    "gfs_edge_gather_stats": [_p, _p, _i, _i, _i, _p, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p],
    "gfs_edge_scatter": [_p, _p, _i, _i, _i, _p, _p],
    "gfs_max_over_k_fwd": [_p, _i, _i64, _i, _p, _i64, _p, _p],
    "gfs_max_over_k_bwd": [_p, _i64, _p, _i, _i64, _i, _p, _p],
    "gfs_softmax_rows_fwd": [_p, _i64, _i, _f, _p, _u32, _f, _p, _p, _p],
    "gfs_softmax_rows_bwd": [_p, _p, _p, _u32, _f, _i64, _i, _f, _p, _p],
    "gfs_dropout_mask": [_i64, _i, _u32, _f, _p, _p],
}
UTILITIES = {"gfs_version": (_i, []), "gfs_last_error_string": (ctypes.c_char_p, []),
             "gfs_device_sm_count": (_i, []), "gfs_set_pdl": (_i, [_i]), "gfs_kmeans_partials": (_i, []),
             "gfs_kmeans_inertia_partials": (_i, []),
             "gfs_knn_tc_workspace_bytes": (_i64, [_i, _i, _i]),
             "gfs_knn_tc_chains": (_i, [_i, _i, _i]), "gfs_knn_tc_set_split": (_i, [_i]),
             "gfs_rowsel_tc_workspace_bytes": (_i64, [_i64, _i]),
             "gfs_rowsel_tc_workspace_bytes_kp": (_i64, [_i64, _i, _i, _i]),
             "gfs_kmeans_accumulate_ranges": (_i, [_i, _i, _i])}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python gfs-3dseg_gws_b200/build.py` "
                "(there is no CPU or PyTorch fallback for the hot path)")
        l = ctypes.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(l, name, None)     # a missing export surfaces as AttributeError at the call site
            if fn is not None:
                fn.restype = _i
                fn.argtypes = args
        for name, (res, args) in UTILITIES.items():
            fn = getattr(l, name, None)
            if fn is not None:
                fn.restype = res
                fn.argtypes = args
        _lib = l
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().gfs_last_error_string().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (gfs_status {rc}): {msg}")
