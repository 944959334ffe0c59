"""ctypes binding of libpn2_b200.so (the C ABI declared in include/pn2_abi.h).

There is deliberately no fallback: if the CUDA library is missing or a call fails, an exception
is raised.  PyTorch is used only for device memory and streams.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(_HERE), "csrc")
LIB_PATH = os.path.join(CSRC, "libpn2_b200.so")

PN2_MAX_LAYERS = 6
REDUCE_MAX, REDUCE_FIRST = 0, 1
ORDER_XYZ_FIRST, ORDER_FEAT_FIRST = 0, 1
ROWS_GROUPED, ROWS_INTERP, ROWS_ALL = 1, 2, 3
FLAG_IN_BF16, FLAG_SKIP_BF16, FLAG_OUT_BF16, FLAG_OUT_ARGMAX = 1, 2, 4, 8

_c_int, _c_float, _vp = ctypes.c_int, ctypes.c_float, ctypes.c_void_p


class Pn2Mlp(ctypes.Structure):
    """struct pn2_mlp (include/pn2_abi.h)"""
    _fields_ = [("num_layers", _c_int),
                ("cin", _c_int * PN2_MAX_LAYERS),
                ("cout", _c_int * PN2_MAX_LAYERS),
                ("relu", _c_int * PN2_MAX_LAYERS),
                ("weight", _vp * PN2_MAX_LAYERS),
                ("bias", _vp * PN2_MAX_LAYERS)]


class Pn2Rows(ctypes.Structure):
    """struct pn2_rows (include/pn2_abi.h)"""
    _fields_ = [("kind", _c_int), ("order", _c_int),
                ("b", _c_int), ("n", _c_int), ("m", _c_int), ("k", _c_int), ("d", _c_int), ("d_skip", _c_int),
                ("xyz", _vp), ("new_xyz", _vp), ("feat", _vp), ("skip", _vp), ("idx", _vp), ("weight", _vp)]


_ROWS = ctypes.POINTER(Pn2Rows)

# name -> argtypes; every function returns int (pn2_status) unless listed in _OTHER
_SIGNATURES = {
    "pn2_furthest_point_sampling": [_c_int, _c_int, _c_int, _vp, _vp, _vp, _vp],
    "pn2_fps_gather": [_c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "pn2_gather_points": [_c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp],
    "pn2_gather_points_grad": [_c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp],
    "pn2_ball_query": [_c_int, _c_int, _c_int, _c_float, _c_int, _vp, _vp, _vp, _vp],
    "pn2_group_points": [_c_int, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp],
    "pn2_group_points_grad": [_c_int, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp],
    "pn2_three_nn": [_c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "pn2_three_interpolate": [_c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "pn2_three_interpolate_grad": [_c_int, _c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "pn2_sphere_iou": [_c_int, _c_int, _vp, _vp, _vp, _vp],
    "pn2_sphere_nms": [_c_int, _c_int, _vp, _vp, _vp, _c_float, _vp, _vp, _vp],
    "pn2_lift_setup": [_c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "pn2_voxel_first_index": [_c_int, _c_int, _vp, _vp, _c_float, _vp, _vp, _vp, _vp, _vp],
    "pn2_label_counts": [_c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "pn2_inverse_index": [_c_int, _c_int, ctypes.c_longlong, _vp, _vp, _vp, _vp],
    "pn2_scatter_rows_det": [_c_int, _c_int, _c_int, ctypes.c_longlong, _c_int, _vp, _vp, _vp, _vp, _vp, _vp],
    "pn2_scatter_rows_det_cl": [_c_int, _c_int, _c_int, ctypes.c_longlong, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "pn2_lift_views": [_c_int] * 6 + [_vp] * 7 + [ctypes.POINTER(_c_float)] + [_c_float] * 3 + [_c_int] + [_vp] * 4,
    "pn2_lift_views_poses": [_c_int] * 6 + [_vp] * 4 + [ctypes.POINTER(_c_float)] * 2 + [_c_float] * 3 + [_c_int] + [_vp] * 4,
    "pn2_lift_views_grad": [_c_int] * 6 + [_vp, _vp, _c_int, _vp, _vp, _vp],
    "pn2_frustum_count": [_c_int, _c_int, _vp, _vp, _vp, _vp, _vp, _vp],
    "pn2_sa_mlp_max": [_c_int] * 5 + [_vp] * 4 + [_c_int, ctypes.POINTER(Pn2Mlp), _vp, _c_int, _c_int, _vp],
    "pn2_fp_mlp": [_c_int] * 5 + [_vp] * 4 + [ctypes.POINTER(Pn2Mlp), _vp, _vp],
    "pn2_sa_all_mlp_max": [_c_int] * 3 + [_vp] * 2 + [ctypes.POINTER(Pn2Mlp), _vp, _c_int, _c_int, _vp],
    "pn2_mlp_pack_bf16": [ctypes.POINTER(Pn2Mlp), _c_int, _vp, _vp],
    "pn2_sa_mlp_max_bf16": [_c_int] * 5 + [_vp] * 4 + [ctypes.POINTER(Pn2Mlp), _vp, _vp, _c_int, _c_int, _c_int, _vp],
    "pn2_fp_mlp_bf16": [_c_int] * 5 + [_vp] * 4 + [ctypes.POINTER(Pn2Mlp), _vp, _vp, _vp, _c_int, _vp],
    "pn2_grid_build": [_c_int, _c_int, _vp, _c_float, _vp, _vp, _vp, _vp, _vp],
    "pn2_ball_query_grid": [_c_int, _c_int, _c_int, _c_float, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "pn2_three_nn_grid": [_c_int, _c_int, _c_int] + [_vp] * 10,
    "pn2_three_nn_weights": [_c_int, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "pn2_transpose": [_c_int, _c_int, _c_int, _vp, _vp, _vp],
    "pn2_train_linear_fwd": [ctypes.c_longlong, _c_int, _c_int] + [_vp] * 8,
    "pn2_train_bn_finalize": [ctypes.c_longlong, _c_int, _vp, _vp, _vp, ctypes.c_double, ctypes.c_double] + [_vp] * 6,
    "pn2_train_bn_bwd_coeffs": [ctypes.c_longlong, _c_int] + [_vp] * 7,
    "pn2_train_bn_running": [_c_int] + [_vp] * 4 + [ctypes.c_double] + [_vp] * 4,
    "pn2_train_bn_running_bwd_coeffs": [_c_int] + [_vp] * 8,
    "pn2_train_bn_relu": [ctypes.c_longlong, _c_int] + [_vp] * 5,
    "pn2_train_bn_bwd_reduce": [ctypes.c_longlong, _c_int] + [_vp] * 6,
    "pn2_train_linear_bwd": [ctypes.c_longlong, _c_int, _c_int] + [_vp] * 14,
    "pn2_train_linear_fwd_rows": [ctypes.c_longlong, _c_int, _c_int, _ROWS] + [_vp] * 5,
    "pn2_train_linear_bwd_rows": [ctypes.c_longlong, _c_int, _c_int, _ROWS] + [_vp] * 12,
    "pn2_train_bn_relu_max": [ctypes.c_longlong, _c_int, _c_int] + [_vp] * 4 + [_c_int, _c_int, _vp, _vp],
    "pn2_train_max_bwd": [ctypes.c_longlong, _c_int, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "pn2_train_bn_relu_max_all": [ctypes.c_longlong, ctypes.c_longlong, _c_int] + [_vp] * 4 + [_c_int, _c_int, _vp, _vp],
    "pn2_train_max_bwd_all": [ctypes.c_longlong, ctypes.c_longlong, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "pn2_scene_index": [_c_int] + [_vp] * 5,
    "pn2_scene_keep": [_c_int, ctypes.c_ulonglong] + [_vp] * 6,
    "pn2_scene_sample": [_c_int] * 4 + [ctypes.c_ulonglong, _c_int] + [_vp] * 4 + [_c_int] + [_vp] * 9,
    "pn2_scene_chunks": [_c_int] + [_vp] * 4,
    "pn2_scene_chunk_rows": [_c_int] * 5 + [_vp] * 10,
    "pn2_scene_votes": [_c_int, _c_int, _vp, _vp, _vp, _c_int, _c_int, _vp, _vp, _vp],
    "pn2_scene_bank_bounds": [_c_int, ctypes.c_longlong, _vp, _vp, _vp, _vp],
    "pn2_scene_crops": [_c_int, ctypes.c_longlong, _c_int, _c_int] + [_vp] * 5 + [_c_int, _vp, _c_int, ctypes.c_ulonglong, _vp, _vp,
                                                                                  _c_int] + [_vp] * 8,
}
_OTHER = {
    "pn2_last_error": ([], ctypes.c_char_p),
    "pn2_abi_version": ([], _c_int),
    "pn2_launch_count": ([], ctypes.c_uint64),
    "pn2_mlp_bf16_supported": ([ctypes.POINTER(Pn2Mlp)], _c_int),
    "pn2_mlp_fp32_supported": ([ctypes.POINTER(Pn2Mlp), _c_int, _c_int], _c_int),
    "pn2_grid_max_points": ([], _c_int),
    "pn2_grid_table_stride": ([], _c_int),
    "pn2_set_fps_policy": ([_c_int], _c_int),
    "pn2_debug_set_fps_mode": ([_c_int], None),
    "pn2_debug_set_tc_timestamps": ([_vp], None),
    "pn2_debug_set_tc_max_ctas": ([_c_int], None),
    "pn2_debug_set_tc_workers": ([_c_int], None),
    "pn2_debug_last_tc_launch": ([ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(_c_int), ctypes.POINTER(_c_int)], _c_int),
    "pn2_debug_set_interp_mode": ([_c_int], None),
    "pn2_mlp_pack_bf16_size": ([ctypes.POINTER(Pn2Mlp)], ctypes.c_longlong),
}

EXPORTS = sorted(list(_SIGNATURES) + list(_OTHER))

_lib = None


class Pn2Error(RuntimeError):
    pass


def load():
    """Loads the shared library (no CUDA call is made)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Pn2Error("libpn2_b200.so not found at %s -- run `python __graft_entry__.py` (build()) or "
                           "`python %s/build.py`; there is no CPU fallback" % (LIB_PATH, CSRC))
        lib = ctypes.CDLL(LIB_PATH)
        for name, argtypes in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = _c_int
        for name, (argtypes, restype) in _OTHER.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = lib
    return _lib


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device=None):
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise Pn2Error("pn2_b200 operators need CUDA tensors (got a %s tensor); there is no CPU path" % t.device)


def check_f32(t, name="tensor", allow_bf16=False):
    """The kernels read raw device pointers as contiguous fp32 (bf16 where stated): anything else would be reinterpreted
    silently, so it is refused here -- the reference raises a dtype error in the same situation."""
    if t is None:
        return None
    require_cuda(t)
    if t.dtype != torch.float32 and not (allow_bf16 and t.dtype == torch.bfloat16):
        raise Pn2Error("%s must be float32%s (got %s)" % (name, " or bfloat16" if allow_bf16 else "", t.dtype))
    return t.contiguous()


def check_i32(t, name="index tensor"):
    if t is None:
        return None
    require_cuda(t)
    if t.dtype != torch.int32:
        raise Pn2Error("%s must be int32 (got %s)" % (name, t.dtype))
    return t.contiguous()


PROFILE = None  # developer profiling: list of (name, start_event, end_event) when enabled


def call(name, *args):
    """Invokes an ABI entry point and raises Pn2Error on a non-zero status."""
    lib = load()
    if PROFILE is not None:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        status = getattr(lib, name)(*args)
        b.record()
        PROFILE.append((name, a, b))
    else:
        status = getattr(lib, name)(*args)
    if status != 0:
        msg = lib.pn2_last_error().decode("utf-8", "replace")
        raise Pn2Error("%s failed with status %d: %s" % (name, status, msg))


def launch_count():
    return int(load().pn2_launch_count())
