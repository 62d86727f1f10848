"""ctypes binding of libxfeat_sm100.so (include/xfeat_b200.h).  No CPU fallback: a missing library is an error."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxfeat_sm100.so")
_lib = None
ABI_VERSION = 2      # XFEAT_ABI_VERSION of include/xfeat_b200.h
N_OVERFLOW = -1      # XF_N_OVERFLOW

c_i, c_f, c_p, c_sz, c_i64 = C.c_int, C.c_float, C.c_void_p, C.c_size_t, C.c_int64

# name -> (restype, argtypes); mirrors include/xfeat_b200.h declaration by declaration
SIGNATURES = {
    "xfeat_abi_version": (c_i, []),
    "xfeat_last_error": (C.c_char_p, []),
    "xfeat_launch_count": (C.c_ulonglong, []),
    "xfeat_packed_weight_floats": (c_sz, []),
    "xfeat_create": (c_i, [C.POINTER(c_p), c_i, c_p, c_sz]),
    "xfeat_destroy": (None, [c_p]),
    "xfeat_resize_bilinear": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i64, c_i64, c_i64, c_i64, c_i, c_p, c_i, c_i, c_f, c_f, c_p]),
    "xfeat_preprocess": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i64, c_i64, c_i64, c_i64, c_i, c_i, c_i, c_p, c_p, c_p]),
    "xfeat_preprocess_scaled": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i64, c_i64, c_i64, c_i64, c_i, c_i, c_i, c_f, c_f, c_p, c_p, c_p]),
    "xfeat_set_conv_impl": (None, [c_i]),
    "xfeat_set_halo_desc_mode": (None, [c_i]),
    "xfeat_get_conv_impl": (c_i, []),
    "xfeat_set_block1_fused": (None, [c_i]),
    "xfeat_get_block1_fused": (c_i, []),
    "xfeat_net_workspace_bytes": (c_sz, [c_i, c_i, c_i]),
    "xfeat_net": (c_i, [c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_sparse_workspace_bytes": (c_sz, [c_i, c_i, c_i, c_i]),
    "xfeat_detect_sparse": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_detect_sparse_split": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_sz, c_p]),
    "xfeat_dense_workspace_bytes": (c_sz, [c_i, c_i, c_i, c_i]),
    "xfeat_detect_dense": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_f, c_f, c_f, c_f, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_set_mnn_impl": (None, [c_i]),
    "xfeat_get_mnn_impl": (c_i, []),
    "xfeat_mnn_workspace_bytes": (c_sz, [c_i, c_i, c_i]),
    "xfeat_mnn_match": (c_i, [c_p, c_p, c_i, c_i64, c_p, c_p, c_i, c_i64, c_i, c_f, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_mnn_match_bounded": (c_i, [c_p, c_p, c_i, c_i64, c_p, c_p, c_i, c_i64, c_i, c_f, c_f, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_mnn_presplit_workspace_bytes": (c_sz, [c_i, c_i, c_i]),
    "xfeat_mnn_match_presplit": (c_i, [c_p, c_p, c_i, c_p, c_p, c_i, c_i, c_i, c_i, c_f, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_gather_matches": (c_i, [c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_i, c_p, c_p, c_p]),
    "xfeat_refine_workspace_bytes": (c_sz, [c_i, c_i]),
    "xfeat_refine": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_f, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_kpts_heatmap": (c_i, [c_p, c_i, c_i, c_i, c_f, c_p, c_p]),
    "xfeat_nms_workspace_bytes": (c_sz, [c_i, c_i, c_i]),
    "xfeat_nms_count": (c_i, [c_p, c_i, c_i, c_i, c_i, c_f, c_p, c_p, c_sz, c_p]),
    "xfeat_nms_write": (c_i, [c_p, c_i, c_i, c_i, c_i, c_f, c_p, c_i, c_p, c_sz, c_p]),
    "xfeat_interpolate_sparse": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p]),
    "xfeat_subpix_softmax2d": (c_i, [c_p, c_i64, c_f, c_p, c_p]),
    "xfeat_fine_matcher_workspace_bytes": (c_sz, [c_i]),
    "xfeat_fine_matcher": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz, c_p]),
    "xfeat_ransac_workspace_bytes": (c_sz, [c_i, c_i]),
    "xfeat_ransac_homography": (c_i, [c_p, c_p, c_p, c_i, c_i, c_f, c_i, C.c_uint32, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_ransac_essential": (c_i, [c_p, c_p, c_p, c_i, c_i, c_f, c_i, C.c_uint32, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "xfeat_debug_conv_layer": (c_i, [c_p, c_i, c_p, c_i, c_i, c_i, c_p, c_p]),
    "xfeat_debug_conv_layer_tc": (c_i, [c_p, c_i, c_p, c_i, c_i, c_i, c_p, c_p, c_sz, c_p]),
    "xfeat_debug_block1_tail": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_sz, c_p]),
}


class XFeatLibraryError(RuntimeError):
    pass


def load():
    """Load the shared library and bind every declared symbol. Raises if the .so or a symbol is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise XFeatLibraryError(
            f"{LIB_PATH} not found: build it with `python -m accelerated_features_b200.build` "
            "(there is no CPU / PyTorch fallback for the XFeat hot path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.xfeat_abi_version() != ABI_VERSION:
        raise XFeatLibraryError(f"ABI version mismatch: library {lib.xfeat_abi_version()} != binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().xfeat_last_error().decode(errors="replace")
        raise XFeatLibraryError(f"{what} failed (code {rc}): {msg}")
