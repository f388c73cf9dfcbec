"""ctypes binding of libflowb200.so (include/flowb200.h).  No CPU fallback: a missing library is an error.

The shared library is built in-tree by `make` / `__graft_entry__.build()` with
`nvcc -gencode arch=compute_100a,code=sm_100a`; it has no torch dependency.  PyTorch is used above
this layer only for device memory and streams.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libflowb200.so")

OK, EINVAL, EWORKSPACE, ECUDA, EUNSUPPORTED = 0, -1, -2, -3, -4
BCD_FP64_F32COST, BCD_FP64_F64COST, BCD_INT32, BCD_INT32_F32COST = 0, 1, 2, 3
BCD_MRF = 16   # OR'd into a BCD mode: block coordinate descent on the MRF energy (include/flowb200.h)
KNN_EXACT_FP64, KNN_TCGEN05 = 0, 1


class CParams(C.Structure):
    """struct flowb200_params (include/flowb200.h)."""
    _fields_ = [
        ("H", C.c_int32), ("W", C.c_int32), ("cellw", C.c_int32), ("cellh", C.c_int32),
        ("cell_radius", C.c_int32), ("k_cell", C.c_int32), ("n_gauss", C.c_int32), ("sigma", C.c_float),
        ("maxnprop", C.c_int32), ("tphi", C.c_float), ("tpsi", C.c_int32), ("lamda", C.c_double),
        ("cost_shift", C.c_int32), ("bcd_mode", C.c_int32), ("knn_mode", C.c_int32), ("con_tresh", C.c_float),
        ("cell_x0", C.c_int32), ("cell_x1", C.c_int32), ("flow_refine", C.c_int32),
    ]


class FlowB200Error(RuntimeError):
    pass


# every symbol include/flowb200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_PP = C.POINTER(CParams)
SYMBOLS = {
    "flowb200_version": (C.c_int, []),
    "flowb200_error_string": (C.c_char_p, [C.c_int]),
    "flowb200_last_cuda_error": (C.c_char_p, []),
    "flowb200_launch_count": (C.c_longlong, []),
    "flowb200_daisy_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "flowb200_daisy": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, C.c_size_t, _P]),
    "flowb200_knn_workspace_bytes": (C.c_size_t, [_PP]),
    "flowb200_knn_proposals": (C.c_int, [_P, _P, _PP, _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "flowb200_knn_debug_scores": (C.c_int, [_P, _P, _PP, _P, _P, _P, C.c_size_t, _P]),
    "flowb200_random_proposals": (C.c_int, [_P, _P, _PP, _P, _P, _P, _P, _P, C.c_uint64, _P]),
    "flowb200_ksets_pack": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "flowb200_quantise_costs": (C.c_int, [_P, _P, C.c_size_t, C.c_double, C.c_int, _P]),
    "flowb200_bcd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "flowb200_bcd_min_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "flowb200_bcd": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int,
                               C.c_int, _P, _P, C.c_size_t, _P]),
    "flowb200_bcd_prepare": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int,
                                       C.c_int, C.c_int, _P, C.c_size_t, _P]),
    "flowb200_bcd_phase": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_int, _P, C.c_size_t, _P]),
    "flowb200_energy": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int,
                                  _P, _P]),
    "flowb200_best_labels": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "flowb200_slot_copy": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, C.c_int, _P, C.c_int, _P]),
    "flowb200_flow_from_labels": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "flowb200_flow_subpixel": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "flowb200_consistency": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "flowb200_segments_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "flowb200_remove_small_segments": (C.c_int, [_P, C.c_int, C.c_int, C.c_float, C.c_int, _P, C.c_size_t, _P]),
    "flowb200_edges_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "flowb200_canny_edges": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_size_t, _P]),
    "flowb200_epe": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_float, _P, _P]),
    "flowb200_pair_workspace_bytes": (C.c_size_t, [_PP]),
    "flowb200_flow_pair": (C.c_int, [_P, _P, _PP, C.c_int, C.c_int, C.c_uint64, _P, _P, _P, _P, C.c_size_t, _P]),
    "flowb200_ctx_create": (_P, [_PP]),
    "flowb200_ctx_destroy": (None, [_P]),
    "flowb200_ctx_flow_pair_host": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_uint64, _P]),
    "flowb200_ctx_flow_pairs_host": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_uint64, _P]),
    "flowb200_consistency_host": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int]),
    "flowb200_remove_small_segments_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_float, C.c_int]),
    "flowb200_canny_edges_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
}

_lib = None


def load():
    """Load libflowb200.so once and declare the prototypes.  Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise FlowB200Error(
            f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
            "There is no CPU fallback for the flow hot path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)      # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc == OK:
        return
    lib = load()
    msg = lib.flowb200_error_string(rc).decode()
    if rc == ECUDA:
        msg += " (" + lib.flowb200_last_cuda_error().decode() + ")"
    raise FlowB200Error(f"{what}: {msg}")
