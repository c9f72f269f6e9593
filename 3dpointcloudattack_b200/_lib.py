"""ctypes binding of libpcdist.so -- the C ABI declared in include/pcdist.h.

There is no fallback of any kind: if the library has not been built, or a call returns a
non-zero status, a RuntimeError is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PCDIST_LIBRARY selects another build of the same ABI (development variants built by tools/)
LIB_PATH = os.environ.get("PCDIST_LIBRARY") or os.path.join(_HERE, "libpcdist.so")

FORM_ROW_COL, FORM_COL_ROW, FORM_SUM_FIRST = 0, 1, 2
NORM_MULSUM, NORM_FMA = 0, 1
VALUE_SQUARED, VALUE_SQRT_CLAMP = 0, 1
KNN_MAX_K, KNN_MAX_C = 64, 128
SOR_MAX_K = 15
SAMPLE_MAX_N = 16384
EDGE_CENTER, EDGE_NEIGHBOR, EDGE_DIFF = 0, 1, 2

_c = ctypes
_P, _I, _L, _F, _Z = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_float, _c.c_size_t
_CLOUD = [_P, _L, _L, _L]

# name -> (restype, argtypes); must list every symbol include/pcdist.h declares
SIGNATURES = {
    "pcd_version": (_I, []),
    "pcd_last_error": (_c.c_char_p, []),
    "pcd_nn1_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "pcd_nn1_query_tiling": (_I, [_I, _I, _I, _c.POINTER(_I), _c.POINTER(_I)]),
    "pcd_nn1_forward": (_I, _CLOUD + _CLOUD + [_I, _I, _I, _I, _I, _I, _I, _F, _F, _P, _P, _P, _P, _P, _P,
                                               _P, _Z, _P, _Z, _P, _Z, _I, _I, _I, _P, _P, _P]),
    "pcd_nn1_backward": (_I, _CLOUD + _CLOUD + [_I, _I, _I, _I, _I] + [_P] * 12 + [_c.POINTER(_L), _F, _F] + _CLOUD + _CLOUD + [_I, _P]),
    "pcd_knn_workspace_bytes": (_Z, [_I, _I, _I, _I, _I]),
    "pcd_knn_forward": (_I, _CLOUD + _CLOUD + [_I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _Z, _I, _P]),
    "pcd_knn_backward": (_I, _CLOUD + _CLOUD + [_I, _I, _I, _I, _I, _P, _P] + _CLOUD + _CLOUD + [_P]),
    "pcd_ball_query": (_I, _CLOUD + _CLOUD + [_I, _I, _I, _F, _I, _P, _P]),
    "pcd_edge_feature_forward": (_I, [_P, _P, _I, _I, _I, _I, _I, _c.POINTER(_I), _P, _P]),
    "pcd_clip_points": (_I, [_P, _P, _P, _I, _I, _I, _c.c_float, _P]),
    "pcd_lp_clip": (_I, [_P, _I, _I, _c.c_float, _P, _P]),
    "pcd_offset_proj": (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "pcd_find_offset": (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "pcd_edge_feature_backward_workspace": (_c.c_size_t, [_I, _I, _I, _I]),
    "pcd_edge_feature_backward": (_I, [_P, _P, _I, _I, _I, _I, _I, _c.POINTER(_I), _P, _P, _c.c_size_t, _P]),
    "pcd_fps": (_I, [_P, _L, _L, _L, _I, _I, _I, _P, _P, _P]),
    "pcd_knn_outlier_forward": (_I, [_P, _I, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P]),
    "pcd_knn_outlier_backward": (_I, _CLOUD + [_P, _P, _P, _L, _I, _I, _I, _I, _P, _I, _P]),
    "pcd_local_frames": (_I, _CLOUD + [_P, _I, _I, _I, _I] + _CLOUD + [_P, _P, _P]),
    "pcd_kappa_forward": (_I, _CLOUD + _CLOUD + [_P, _P, _I, _I, _I, _I, _P, _P]),
    "pcd_kappa_backward": (_I, _CLOUD + _CLOUD + [_P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "pcd_graph_laplacian": (_I, _CLOUD + [_P, _I, _I, _I, _P, _P]),
    "pcd_sor_forward": (_I, _CLOUD + [_I, _I, _I, _c.c_double, _P, _P, _P, _P, _P, _P]),
    "pcd_sor_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "pcd_sor_forward_len": (_I, _CLOUD + [_I, _I, _I, _c.c_double, _P, _I, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "pcd_nn_dist64_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "pcd_nn_dist64_forward": (_I, _CLOUD + _CLOUD + [_I, _I, _I, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "pcd_sample_points": (_I, [_I, _I, _I, _P, _P, _L, _c.c_uint64, _L, _P, _P, _P]),
    "pcd_fp32_probe_launch": (_I, [_I, _I, _P, _c.POINTER(_c.c_double), _P]),
}

_lib = None


def load():
    """Load libpcdist.so and declare every prototype. Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python 3dpointcloudattack_b200/build.py` "
            "(or __graft_entry__.build()). There is no CPU / PyTorch fallback for this path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)     # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what):
    if status != 0:
        msg = load().pcd_last_error()
        raise RuntimeError(f"{what} failed with status {status}: {msg.decode() if msg else ''}")
