"""ctypes binding of libl3d_b200.so (the C ABI declared in include/l3d_b200.h).

There is NO fallback: if the CUDA library is missing or a tensor is not a CUDA fp32 tensor the
call raises.  PyTorch is used only for device memory and streams.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# L3D_B200_LIB loads another build of the same library instead of the in-tree one, e.g. a parent commit's
# build for an A/B comparison of bench.py runs
LIB_PATH = os.environ.get("L3D_B200_LIB") or os.path.join(_HERE, "libl3d_b200.so")
_lib = None

_P = ctypes.c_void_p
_I = ctypes.c_int
_F = ctypes.c_float

# name -> argtypes (all return int unless listed in _RESTYPE)
_SIGNATURES = {
    "l3d_abi_version": [],
    "l3d_error_string": [_I],
    "l3d_launch_count": [],
    "l3d_debug_force_slow_path": [_I],
    "l3d_debug_knn_path": [_I],
    "l3d_knn_expansion": [_P, _I, _I, _I, _P, _P, _P],
    "l3d_knn_expansion_host": [_P, _I, _I, _I, _P],
    "l3d_knn_graph_feature": [_P, _I, _I, _I, _P, _P, _P],
    "l3d_knn_features_ws_bytes": [_I, _I, _I],
    "l3d_knn_features": [_P, _I, _I, _I, _I, _P, _P, _P],
    "l3d_graph_feature": [_P, _P, _I, _I, _I, _I, _P, _P],
    "l3d_graph_feature_grad": [_P, _P, _I, _I, _I, _I, _P, _P],
    "l3d_knn_point": [_P, _P, _I, _I, _I, _I, _P, _P, _P],
    "l3d_knn_sqdist": [_P, _P, _I, _I, _I, _I, _P, _P],
    "l3d_pn2_knn": [_I, _I, _I, _I, _P, _P, _P, _P, _P],
    "l3d_pn2_three_nn": [_I, _I, _I, _P, _P, _P, _P, _P],
    "l3d_pn2_ball_query": [_I, _I, _I, _F, _I, _P, _P, _P, _P],
    "l3d_pn2_group_points": [_I, _I, _I, _I, _I, _P, _P, _P, _P],
    "l3d_pn2_group_points_grad": [_I, _I, _I, _I, _I, _P, _P, _P, _P],
    "l3d_pn2_gather_points": [_I, _I, _I, _I, _P, _P, _P, _P],
    "l3d_pn2_gather_points_grad": [_I, _I, _I, _I, _P, _P, _P, _P],
    "l3d_pn2_furthest_point_sampling": [_I, _I, _I, _P, _P, _P, _P],
    "l3d_pn2_three_interpolate": [_I, _I, _I, _I, _P, _P, _P, _P, _P],
    "l3d_pn2_three_interpolate_grad": [_I, _I, _I, _I, _P, _P, _P, _P, _P],
    "l3d_query_ball_point": [_P, _P, _I, _I, _I, _F, _I, _P, _P, _P, _P],
    "l3d_farthest_point_sample": [_P, _I, _I, _I, _P, _P, _P],
    "l3d_square_distance": [_P, _P, _I, _I, _I, _P, _P],
    "l3d_index_points": [_P, _P, _I, _I, ctypes.c_int64, _I, _P, _P],
    "l3d_index_points_grad": [_P, _P, _I, _I, ctypes.c_int64, _I, _P, _P],
    "l3d_compute_density": [_P, _I, _I, _F, _F, _P, _P],
    "l3d_emd_forward_ws_bytes": [_I, _I, _I],
    "l3d_emd_forward": [_P, _P, _I, _I, _I, _P, _P, _P, _P],
    "l3d_emd_backward_ws_bytes": [_I, _I, _I],
    "l3d_debug_emd_force_multilaunch": [_I],
    "l3d_emd_backward": [_P, _P, _P, _I, _I, _I, _P, _P, _P, _P],
    "l3d_kabsch3x3_batched": [_P, _P, _P, _I, _P, _P, _P],
    "l3d_svd_head_tail": [_P, _P, _I, _I, _P, _P, _P],
    "l3d_svd_head_tail_backward": [_P, _P, _P, _P, _I, _I, _P, _P, _P],
    "l3d_soft_correspondence": [_P, _P, _P, _I, _I, _I, _I, _P, _P],
    "l3d_soft_correspondence_status": [],
    "l3d_debug_soft_correspondence_force_generic": [_I],
    "l3d_debug_soft_correspondence_split": [_I],
    "l3d_debug_soft_correspondence_tiles": [_P],
    "l3d_debug_soft_correspondence_scores": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P],
    "l3d_chamfer_loss_fwd_bwd_host": [_P, _P, _I, _I, _I, _P, _P, _P],
    "l3d_topk_rows": [_P, ctypes.c_longlong, _I, _I, _P, _P],
    "l3d_feature_square_distance_ws_bytes": [_I, _I, _I],
    "l3d_feature_square_distance": [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P],
    "l3d_sinkhorn_ws_bytes": [_I, _I, _I],
    "l3d_sinkhorn": [_P, _I, _I, _I, _I, _I, _P, _P, _P],
    "l3d_rpm_match_tail": [_P, _P, _I, _I, _I, _I, _I, _F, _P, _P, _P, _P, _P],
    "l3d_weighted_rigid_transform": [_P, _P, _P, _I, _I, _F, _P, _P],
    "l3d_edgeconv_layer1": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, ctypes.c_longlong, _I, _P],
    "l3d_conv1x1_bn_relu_maxk": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P, ctypes.c_longlong, _I, _P],
    "l3d_edgeconv_status": [],
    "l3d_soft_correspondence_dscores": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P],
    "l3d_linear_cm": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P],
    "l3d_attention_bounds_ws_bytes": [_I],
    "l3d_attention_bounds": [_P, _P, _I, _I, _I, _I, _P, _P, _P],
    "l3d_attention_stats_if": [_P, _P, _I, _I, _I, _I, _P, _P, _P],
    "l3d_linear_cm_t": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    "l3d_attention_stats": [_P, _P, _I, _I, _I, _I, _I, _P, _P],
    "l3d_attention_probs_t": [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P],
    "l3d_layernorm_cm": [_P, _P, _P, _F, _I, _I, _I, _P, _P],
    "l3d_chamfer_forward": [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P],
    "l3d_chamfer_backward": [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P],
    "l3d_chamfer_ws_bytes": [_I, _I, _I],
    "l3d_chamfer_loss_forward": [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P],
    "l3d_chamfer_loss_backward": [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P],
}
_RESTYPE = {
    "l3d_error_string": ctypes.c_char_p,
    "l3d_launch_count": ctypes.c_uint64,
    "l3d_debug_force_slow_path": None,
    "l3d_debug_knn_path": None,
    "l3d_debug_emd_force_multilaunch": None,
    "l3d_debug_soft_correspondence_force_generic": None,
    "l3d_debug_soft_correspondence_split": None,
    "l3d_chamfer_ws_bytes": ctypes.c_size_t,
    "l3d_knn_features_ws_bytes": ctypes.c_size_t,
    "l3d_emd_forward_ws_bytes": ctypes.c_size_t,
    "l3d_feature_square_distance_ws_bytes": ctypes.c_size_t,
    "l3d_sinkhorn_ws_bytes": ctypes.c_size_t,
    "l3d_attention_bounds_ws_bytes": ctypes.c_size_t,
    "l3d_emd_backward_ws_bytes": ctypes.c_size_t,
}


def exported_symbols():
    """Every symbol include/l3d_b200.h declares (checked by tests/test_abi.py)."""
    return sorted(_SIGNATURES)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "learning3d_b200: %s not found — build it with `make -C learning3d_b200/csrc` "
                "(or __graft_entry__.build()).  There is no CPU fallback." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, argtypes in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = _RESTYPE.get(name, _I)
        _lib = handle
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().l3d_error_string(int(rc))
        raise RuntimeError("learning3d_b200 %s failed: %s (code %d)" % (what, msg.decode(), rc))


def stream():
    return _P(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL = "argument not given").  An EMPTY tensor has a null
    data_ptr; the ABI treats NULL as a missing argument, so empty tensors pass a never-dereferenced
    non-null sentinel and the entry point returns L3D_OK on its `B == 0` early-out."""
    if t is None:
        return _P(None)
    return _P(t.data_ptr() or 16)


def require_cuda(t, name, dtype=torch.float32):
    """The hot path is CUDA-only: never silently compute on the CPU."""
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError("learning3d_b200: %s must be a CUDA tensor (no CPU fallback)" % name)
    if t.dtype != dtype:
        raise TypeError("learning3d_b200: %s must be %s, got %s" % (name, dtype, t.dtype))
    return t.contiguous()


class _NullCtx(object):
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NULL = _NullCtx()


def on_device(dev):
    """Context that makes `dev` current; free when it already is (torch.cuda.device costs ~10 us)."""
    if dev.index is None or dev.index == torch.cuda.current_device():
        return _NULL
    return torch.cuda.device(dev)


def launch_count():
    return int(lib().l3d_launch_count())
