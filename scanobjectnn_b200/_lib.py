"""ctypes binding of libpsa.so (the C ABI declared in include/psa.h).

There is NO fallback: if the CUDA library is missing or fails to load, importing any op raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PSA_LIB_PATH") or os.path.join(_HERE, "libpsa.so")   # PSA_LIB_PATH: instrumented builds of tools/

PSA_MAX_MLP_LAYERS = 4


class PsaError(RuntimeError):
    """Raised for PSA_ERR_UNSUPPORTED or a failed CUDA launch."""


class PsaMlp(C.Structure):
    _fields_ = [
        ("n_layers", C.c_int),
        ("channels", C.c_int * (PSA_MAX_MLP_LAYERS + 1)),
        ("weight", C.c_void_p * PSA_MAX_MLP_LAYERS),
        ("scale", C.c_void_p * PSA_MAX_MLP_LAYERS),
        ("shift", C.c_void_p * PSA_MAX_MLP_LAYERS),
        ("relu", C.c_int * PSA_MAX_MLP_LAYERS),
        ("image", C.c_void_p * PSA_MAX_MLP_LAYERS),
        ("image_nt", C.c_int * PSA_MAX_MLP_LAYERS),
        ("image_row0", C.c_int * PSA_MAX_MLP_LAYERS),
    ]


class PsaActIn(C.Structure):
    """psa_act_in (include/psa.h): forward input of a training-mode layer."""
    _fields_ = [("x", C.c_void_p), ("ld", C.c_longlong), ("scale", C.c_void_p), ("shift", C.c_void_p), ("mask", C.c_void_p),
                ("relu", C.c_int)]


class PsaGradIn(C.Structure):
    """psa_grad_in (include/psa.h): gradient w.r.t. a layer's pre-batch-norm output, evaluated on the fly."""
    _fields_ = [("y", C.c_void_p), ("ld", C.c_longlong), ("s", C.c_void_p), ("t", C.c_void_p), ("relu", C.c_int),
                ("ca", C.c_void_p), ("cb", C.c_void_p), ("cc", C.c_void_p), ("dh", C.c_void_p), ("ld_dh", C.c_longlong),
                ("mask", C.c_void_p), ("dp", C.c_void_p), ("pv", C.c_void_p), ("argk", C.c_void_p), ("pool_k", C.c_int),
                ("C", C.c_int), ("mode", C.c_int)]


_i, _f, _p = C.c_int, C.c_float, C.c_void_p
_ll, _sz = C.c_longlong, C.c_size_t
_ain, _gin = C.POINTER(PsaActIn), C.POINTER(PsaGradIn)

# name -> argtypes; every entry point returns int.  Mirrors include/psa.h one to one
# (tests/test_abi.py checks header <-> this table <-> exported symbols).
SIGNATURES = {
    "psa_farthest_point_sample": [_i, _i, _i, _p, _p, _p, _p],
    "psa_gather_point": [_i, _i, _i, _p, _p, _p, _p],
    "psa_gather_point_grad": [_i, _i, _i, _p, _p, _p, _p, _sz, _p],
    "psa_query_ball_point": [_i, _i, _i, _f, _i, _p, _p, _p, _p, _p],
    "psa_group_point": [_i, _i, _i, _i, _i, _p, _p, _p, _p],
    "psa_group_point_grad": [_i, _i, _i, _i, _i, _p, _p, _p, _p, _sz, _p],
    "psa_selection_sort": [_i, _i, _i, _i, _p, _p, _p, _p],
    "psa_knn_point": [_i, _i, _i, _i, _i, _p, _p, _p, _p, _p],
    "psa_three_nn": [_i, _i, _i, _p, _p, _p, _p, _p],
    "psa_three_interpolate": [_i, _i, _i, _i, _p, _p, _p, _p, _p],
    "psa_three_interpolate_grad": [_i, _i, _i, _i, _p, _p, _p, _p, _p, _sz, _p],
    "psa_three_nn_interpolate": [_i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p],
    "psa_augment_batch": [_i, _i, _i, _p, _p, _p, _p, _p, _p, C.c_double, C.c_double, _p, _i, _i, _p, _p],
    "psa_pairwise_distance": [_i, _i, _i, _p, _p, _p],
    "psa_knn_topk": [_i, _i, _i, _i, _p, _p, _p],
    "psa_knn_graph": [_i, _i, _i, _i, _p, _p, _p],
    "psa_get_edge_feature": [_i, _i, _i, _i, _p, _p, _p, _p],
    "psa_knn_graph_ws": [_i, _i, _i, _i, _p, _p, _p, C.c_size_t, _p],
    "psa_shared_mlp": [C.c_longlong, _i, _p, C.POINTER(PsaMlp), _p, _p, C.c_size_t, _p],
    "psa_sa_module_infer": [_i, _i, _i, _i, _f, _i, _p, _p, _p, _p, C.POINTER(PsaMlp), _p, _p, _p, _p, C.c_size_t, _p],
    "psa_sa_conv1_prebn": [_i, _i, _i, _i, _f, _i, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, C.c_size_t, _p],
    "psa_sa_group_all_infer": [_i, _i, _i, _p, _p, C.POINTER(PsaMlp), _p, _p, C.c_size_t, _p],
    "psa_mlp_image_plan": [_i, C.c_longlong, _i, _i, _i, C.POINTER(PsaMlp), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t)],
    "psa_prepare_weight_image": [_i, _i, _i, _i, _p, _p, _p],
    "psa_set_mlp_mode": [_i],
    "psa_get_mlp_mode": [],
    "psa_edgeconv_infer": [_i, _i, _i, _i, _p, _p, C.POINTER(PsaMlp), _p, _p, C.c_size_t, _p],
    # training mode
    "psa_train_dense_fwd": [_ll, _i, _i, _ain, _p, _p, _p, _p, _p, _sz, _p],
    "psa_train_dense_bwd_input": [_ll, _i, _i, _gin, _p, _p, _ll, _i, _p, _sz, _p],
    "psa_train_dense_bwd_weight": [_ll, _i, _i, _ain, _gin, _p, _p, _sz, _p],
    "psa_train_bias_grad": [_ll, _i, _gin, _p, _p],
    "psa_bn_finalize": [_i, _ll, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p],
    "psa_train_pool_fwd": [_ll, _i, _i, _p, _p, _p, _p, _p, _p],
    "psa_bn_bwd_coeffs": [_ll, _i, _gin, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p],
    "psa_sa_conv1_bwd": [_i, _i, _i, _i, _i, _p, _p, _p, _gin, _p, _p, _p, _sz, _p],
    "psa_fp_conv1_prebn": [_i, _i, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _sz, _p],
    "psa_fp_conv1_bwd": [_i, _i, _i, _i, _p, _p, _gin, _p, _p, _sz, _p],
    "psa_cls_seg_xent": [_i, _i, _i, _p, _p, _p, _p, _f, _p, _p, _p, _p, _sz, _p],
    "psa_softmax_xent": [_i, _i, _p, _p, _p, _p, _p],
    "psa_pool_rows": [_ll, _i, _i, _i, _p, _p, _p, _p],
    "psa_adam_step": [_ll, _p, _p, _p, _p, _f, _f, _f, _f, _i, _f, _p],
}
INFO_SYMBOLS = ("psa_version", "psa_last_error", "psa_sm_arch", "psa_shared_mlp_workspace_bytes",
                "psa_sa_module_workspace_bytes", "psa_sa_conv1_prebn_workspace_bytes", "psa_sa_group_all_workspace_bytes", "psa_edgeconv_workspace_bytes",
                "psa_train_dense_workspace_bytes", "psa_bn_bwd_workspace_bytes", "psa_sa_conv1_bwd_workspace_bytes", "psa_knn_graph_workspace_bytes",
                "psa_scatter_workspace_bytes", "psa_fp_conv1_prebn_workspace_bytes", "psa_fp_conv1_bwd_workspace_bytes",
                "psa_cls_seg_xent_workspace_bytes")

_lib = None


def load() -> C.CDLL:
    """Load libpsa.so and bind every entry point.  Raises if the library or a symbol is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m scanobjectnn_b200.build` "
            "(there is no CPU or PyTorch fallback for the point-set-abstraction ops)")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.psa_shared_mlp_workspace_bytes.argtypes = [C.c_longlong, C.POINTER(PsaMlp)]
    lib.psa_shared_mlp_workspace_bytes.restype = C.c_size_t
    lib.psa_sa_module_workspace_bytes.argtypes = [_i, _i, _i, _i, _i, C.POINTER(PsaMlp)]
    lib.psa_sa_module_workspace_bytes.restype = C.c_size_t
    lib.psa_edgeconv_workspace_bytes.argtypes = [_i, _i, _i, _i, C.POINTER(PsaMlp)]
    lib.psa_edgeconv_workspace_bytes.restype = C.c_size_t
    lib.psa_sa_group_all_workspace_bytes.argtypes = [_i, _i, _i, C.POINTER(PsaMlp)]
    lib.psa_sa_group_all_workspace_bytes.restype = C.c_size_t
    lib.psa_sa_conv1_prebn_workspace_bytes.argtypes = [_i, _i, _i, _i, _i, _i]
    lib.psa_sa_conv1_prebn_workspace_bytes.restype = C.c_size_t
    lib.psa_train_dense_workspace_bytes.argtypes = [_ll, _i, _i]
    lib.psa_train_dense_workspace_bytes.restype = C.c_size_t
    lib.psa_bn_bwd_workspace_bytes.argtypes = [_i]
    lib.psa_bn_bwd_workspace_bytes.restype = C.c_size_t
    lib.psa_sa_conv1_bwd_workspace_bytes.argtypes = [_i, _i, _i, _i, _i, _i]
    lib.psa_sa_conv1_bwd_workspace_bytes.restype = C.c_size_t
    lib.psa_knn_graph_workspace_bytes.argtypes = [_i, _i, _i, _i]
    lib.psa_knn_graph_workspace_bytes.restype = C.c_size_t
    lib.psa_scatter_workspace_bytes.argtypes = [_i, _i, _ll]
    lib.psa_scatter_workspace_bytes.restype = C.c_size_t
    for name, argtypes in (("psa_fp_conv1_prebn_workspace_bytes", [_i, _i, _i]), ("psa_fp_conv1_bwd_workspace_bytes", [_i, _i, _i]),
                           ("psa_cls_seg_xent_workspace_bytes", [_i, _i])):
        getattr(lib, name).argtypes = argtypes
        getattr(lib, name).restype = C.c_size_t
    lib.psa_version.restype = C.c_int
    lib.psa_sm_arch.restype = C.c_int
    lib.psa_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    """Map a C-ABI return code onto the reference's error behaviour: InvalidArgument -> ValueError."""
    if rc == 0:
        return
    msg = load().psa_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(msg or what)
    raise PsaError(f"{what}: rc={rc}: {msg}")
