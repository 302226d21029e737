"""ctypes binding of libpcreid_sm100.so (C ABI declared in include/pcreid.h).

The library is the product: if it is missing we try one in-tree build and otherwise raise.  There is
no CPU or PyTorch fallback for any compute entry point.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpcreid_sm100.so")
_lib = None

c_int, c_ll, c_float, c_vp = ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_void_p


class LinearArgs(ctypes.Structure):
    """struct pcreid_linear_args (include/pcreid.h)."""
    _fields_ = [
        ("B", c_int), ("rows", c_int), ("CO", c_int), ("K1", c_int), ("K2", c_int),
        ("X1", c_vp), ("x1_bs", c_ll), ("ldx1", c_int), ("x1_pm", c_int), ("x1_map", c_vp),
        ("X2", c_vp), ("x2_bs", c_ll), ("ldx2", c_int), ("x2_pm", c_int), ("x2_map", c_vp),
        ("W1", c_vp), ("w1_bs", c_ll), ("w1_map", c_vp),
        ("W2", c_vp), ("w2_bs", c_ll),
        ("bias", c_vp),
        ("R", c_vp), ("r_bs", c_ll), ("ldr", c_int), ("r_map", c_vp), ("res_after_act", c_int),
        ("act", c_int),
        ("Y", c_vp), ("y_bs", c_ll), ("ldy", c_int), ("y_pm", c_int),
    ]


class NormArgs(ctypes.Structure):
    """struct pcreid_norm_args (include/pcreid.h)."""
    _fields_ = [
        ("B", c_int), ("rows", c_int), ("C", c_int), ("G", c_int),
        ("X", c_vp), ("x_bs", c_ll), ("ldx", c_int),
        ("gamma", c_vp), ("beta", c_vp),
        ("R", c_vp), ("r_bs", c_ll), ("ldr", c_int), ("r_map", c_vp),
        ("act", c_int),
        ("Y", c_vp), ("y_bs", c_ll), ("ldy", c_int),
    ]


_SIGS = {
    "pcreid_abi_version": [],
    "pcreid_fps": [c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_fps_with_dist": [c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_fps_block_size": [c_int],
    "pcreid_fps_torch": [c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_pairwise_sqdist": [c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_vp],
    "pcreid_knn": [c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_knn_t": [c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_knn_point": [c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_knn_point_set": [c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_knn_feature": [c_int, c_int, c_int, c_int, c_vp, c_ll, c_vp, c_vp],
    "pcreid_ball_query": [c_int, c_int, c_int, c_float, c_float, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_query_ball_point": [c_int, c_int, c_int, c_float, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_group_points": [c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_gather_points": [c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_query_group": [c_int] * 5 + [c_vp] * 4 + [c_int, c_float, c_vp, c_vp, c_vp],
    "pcreid_crop_tiles": [c_int],
    "pcreid_crop_mask": [c_int, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_crop_gather": [c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_crop_mask_scenes": [c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_crop_gather_scenes": [c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_three_nn": [c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_three_interpolate": [c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_cn_linear": [ctypes.POINTER(LinearArgs), c_vp],
    "pcreid_cn_linear_tc": [ctypes.POINTER(LinearArgs), c_vp],
    "pcreid_cn_linear_tc2": [ctypes.POINTER(LinearArgs), c_vp, c_vp, c_int, c_vp],
    "pcreid_cn_linear_tma": [ctypes.POINTER(LinearArgs), c_ll, c_ll, c_ll, c_int, c_int, c_vp],
    "pcreid_cn_linear_tma_x3": [ctypes.POINTER(LinearArgs), c_vp, c_vp, c_ll, c_ll, c_ll, c_int, c_vp],
    "pcreid_cn_groupnorm": [ctypes.POINTER(NormArgs), c_vp],
    "pcreid_gn_res_relu_dot": [c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_float, c_vp, c_vp],
    "pcreid_attn_front_blob_bytes": [c_int, c_int, c_int, c_int],
    "pcreid_attn_front": [c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_ll, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_ll, c_int,
                          c_vp],
    "pcreid_linattn_kv_img": [c_int, c_int, c_int, c_int, c_vp, c_ll, c_int, c_vp, c_ll, c_int, c_vp, c_vp, c_vp],
    "pcreid_attn_back_objects_per_tile": [c_int, c_int],
    "pcreid_attn_back_blob_bytes": [c_int, c_int, c_int, c_int],
    "pcreid_attn_back": [c_int] * 8 + [c_vp, c_ll, c_int, c_vp, c_ll, c_int] + [c_vp] * 7 + [c_vp, c_ll, c_int, c_vp],
    "pcreid_linattn_kv": [c_int, c_int, c_int, c_int, c_vp, c_ll, c_int, c_vp, c_ll, c_int, c_vp, c_vp, c_vp],
    "pcreid_linattn_scale": [c_int, c_int, c_int, c_int, c_int, c_vp, c_ll, c_int, c_vp, c_vp, c_vp, c_vp, c_ll, c_int, c_vp],
    "pcreid_local_linattn": [c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_cn_pool": [c_int, c_int, c_int, c_vp, c_ll, c_int, c_int, c_vp, c_ll, c_int, c_int, c_vp, c_ll, c_ll, c_vp],
    "pcreid_cn_chanmax": [c_int, c_int, c_int, c_vp, c_ll, c_int, c_vp, c_ll, c_ll, c_vp],
    "pcreid_sa_edge_mlp": [c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_edge_build": [c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp],
    "pcreid_seg_max": [c_ll, c_int, c_vp, c_vp, c_vp],
    "pcreid_seg_mean": [c_ll, c_int, c_vp, c_vp, c_vp],
    "pcreid_edge_gather_max": [c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_ll, c_int, c_vp],
    "pcreid_pack_image": [c_int, c_int, c_int, c_vp, c_ll, c_int, c_int, c_int, c_vp, c_vp],
    "pcreid_pack_image_bias": [c_int, c_int, c_int, c_vp, c_ll, c_int, c_vp, c_int, c_vp, c_vp],
    "pcreid_pack_b7": [c_int, c_vp, c_vp, c_int, c_vp, c_vp],
    "pcreid_pool_finish2": [c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "pcreid_pair_p1a2": [c_int, c_int, c_int, c_int, c_float] + [c_vp] * 8 + [c_int, c_vp],
    "pcreid_pair_p1b_n": [c_int, c_int, c_int, c_int, c_float] + [c_vp] * 7 + [c_int, c_vp],
    "pcreid_pair_p2y": [c_int, c_int, c_int, c_int, c_float] + [c_vp] * 5 + [c_int, c_vp],
    "pcreid_sa_edge_mlp_tc": [c_int, c_int, c_int, c_int, c_int] + [c_vp] * 8 + [c_int, c_vp],
    "pcreid_sa_edge_mlp_tc2": [c_int, c_int, c_int, c_int, c_int] + [c_vp] * 8 + [c_int, c_int, c_vp],
    "pcreid_pair_concat_head_tc": [c_int, c_int, c_int, c_int] + [c_vp] * 10 + [c_float, c_vp, c_vp, c_int, c_vp],
    "pcreid_pair_concat_head": [c_int, c_int, c_int, c_int] + [c_vp] * 10 + [c_float, c_vp, c_vp, c_vp],
    "pcreid_lsap_workspace_bytes": [c_int, c_int],
    "pcreid_lsap": [c_int, c_int, c_int, c_vp, c_vp, c_float, c_vp, c_vp, c_vp, c_vp],
    "pcreid_lsap_blocks": [c_int, c_int, c_int, c_vp, c_vp, c_vp, c_float, c_vp, c_vp, c_vp, c_vp],
    "pcreid_track_gate_blocks": [c_int] * 4 + [c_vp] * 8 + [c_int] * 3 + [c_vp, c_vp, c_vp],
    "pcreid_track_update": [c_int] * 3 + [c_vp] * 5 + [c_int, c_int] + [c_vp] * 13 + [c_vp],
    "pcreid_track_scatter": [c_int, c_vp, c_ll, c_vp, c_vp, c_ll, c_vp, c_vp, c_vp],
    "pcreid_track_predict": [c_int] * 3 + [c_vp] * 6 + [c_float, c_float, c_vp],
    "pcreid_track_correct": [c_int] * 3 + [c_vp] * 8 + [c_float] * 3 + [c_vp],
    "pcreid_track_gate_motion_blocks": [c_int] * 4 + [c_vp] * 8 + [c_int] * 3 + [c_vp, c_vp, c_float, c_float, c_vp, c_vp],
}

ERRORS = {1: "PCREID_ERR_ARG (bad pointer/size)", 2: "PCREID_ERR_LAUNCH (CUDA launch failed)",
          3: "PCREID_ERR_UNSUPPORTED (shape outside the built kernels)"}


def exported_symbols():
    return sorted(_SIGS.keys())


def lib():
    """Returns the loaded CDLL; builds it once if absent; raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build
        _build.build_library()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing and could not be built: the CUDA extension is required "
                           "(no CPU fallback exists)")
    L = ctypes.CDLL(LIB_PATH)
    for name, argt in _SIGS.items():
        fn = getattr(L, name)     # AttributeError here == header/library mismatch: fail loudly
        fn.argtypes = argt
        fn.restype = c_int
    _lib = L
    return L


ABI_CALLS = 0   # number of C-ABI compute calls made by this process (each launches >= 1 kernel)


def check(rc, what):
    global ABI_CALLS
    ABI_CALLS += 1
    if rc != 0:
        raise RuntimeError(f"{what} failed: {ERRORS.get(rc, rc)}")
