"""ctypes binding of libpn2_b200.so (include/pn2_b200.h) -- the only native doorway.

PyTorch tensors are used purely as device-memory containers: every call hands raw
``data_ptr()`` addresses plus the current CUDA stream to the C ABI.  There is NO CPU or
PyTorch fallback: if the library is missing, or a tensor is not a contiguous CUDA tensor
of the expected dtype, the call fails loudly.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# PN2_LIB: load another build of the same library (the -DPN2_TRACE diagnostics build); never a fallback
LIB_PATH = os.environ.get("PN2_LIB") or os.path.join(_HERE, "lib", "libpn2_b200.so")

PN2_OK, PN2_EINVAL, PN2_ELAUNCH, PN2_EUNSUPPORTED, PN2_ENULL = 0, -1, -2, -3, -4

_vp, _i, _l, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_float
_ull = ctypes.c_ulonglong

# name -> argument ctypes (return type is always int unless listed in _RESTYPE)
SIGNATURES = {
    "pn2_abi_version": [],
    "pn2_strerror": [_i],
    "pn2_last_cuda_error": [],
    "pn2_set_sm_budget": [_i],
    "pn2_get_sm_budget": [],
    "pn2_ball_threshold": [_f],
    "pn2_fps": [_i, _i, _i, _vp, _vp, _vp, _vp],
    "pn2_fps_cluster": [_i, _i, _i, _vp, _vp, _vp],
    "pn2_fps_cluster_mb": [_i, _i, _i, _vp, _vp, _vp],
    "pn2_cumsum": [_i, _i, _vp, _vp, _vp],
    "pn2_prob_sample": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "pn2_gather_point": [_i, _i, _i, _vp, _vp, _vp, _vp],
    "pn2_gather_point_grad": [_i, _i, _i, _vp, _vp, _vp, _vp],
    "pn2_query_ball_point": [_i, _i, _i, _f, _i, _vp, _vp, _vp, _vp, _vp],
    "pn2_ball_grid_workspace_bytes": [_i, _i],
    "pn2_query_ball_point_grid": [_i, _i, _i, _f, _i, _vp, _vp, _vp, _vp, _vp, _l, _vp],
    "pn2_group_point": [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "pn2_group_point_grad": [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "pn2_three_nn": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "pn2_interpolate_label_with_color": [_i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp],
    "pn2_three_interpolate": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "pn2_three_interpolate_grad": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "pn2_selection_sort": [_i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "pn2_knn_point": [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "pn2_group_concat": [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp],
    "pn2_group_concat_ld": [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _i, _vp],
    "pn2_group_concat_grad": [_i, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp],
    "pn2_fp_weights": [_i, _vp, _vp, _vp],
    "pn2_three_interpolate_ld": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "pn2_three_interpolate_grad_ld": [_i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp],
    "pn2_copy_cols": [_l, _i, _vp, _i, _vp, _i, _i, _vp],
    "pn2_linear_fwd": [_l, _i, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _l, _i, _vp],
    "pn2_linear_fwd_bn": [_l, _i, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _l, _i, _vp],
    "pn2_linear_workspace_bytes": [_i, _i],
    "pn2_linear_image_bytes": [_i, _i, _i],
    "pn2_linear_image_describe": [_i, _i, _i, _vp, _vp, _vp],
    "pn2_linear_prepare": [_i, _vp, _vp],
    "pn2_linear_dgrad": [_l, _i, _i, _vp, _vp, _vp, _i, _vp, _l, _i, _vp],
    "pn2_linear_wgrad": [_l, _i, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp],
    "pn2_bn_train_finalize": [_i, _l, _vp, _vp, _vp, _f, _f, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "pn2_bn_eval_affine": [_i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp],
    "pn2_affine_act": [_l, _i, _vp, _vp, _vp, _i, _vp, _i, _vp],
    "pn2_pool_weights": [_l, _i, _vp, _i, _vp, _vp],
    "pn2_group_pool": [_l, _i, _i, _vp, _vp, _i, _vp, _vp, _vp],
    "pn2_group_pool_grad": [_l, _i, _i, _vp, _vp, _vp, _i, _vp, _vp],
    "pn2_relu_mask": [_l, _i, _vp, _vp, _vp, _vp, _vp],
    "pn2_affine_act_maxpool": [_l, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp],
    "pn2_bn_bwd_reduce": [_l, _i, _vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp],
    "pn2_bn_bwd_apply": [_l, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp,
                         _vp],
    "pn2_bn_bwd_reduce_pool": [_l, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp],
    "pn2_bn_bwd_apply_pool": [_l, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp,
                              _vp, _vp, _vp],
    "pn2_dropout": [_l, _vp, _f, _ull, _vp, _vp, _vp],
    "pn2_dropout_mask": [_l, _f, _ull, _vp, _vp],
    "pn2_softmax_ce_reduce": [_l, _i, _vp, _vp, _vp, _vp, _vp],
    "pn2_softmax_ce_grad": [_l, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp],
    "pn2_sa_workspace_bytes": [_vp, _vp],
    "pn2_sa_forward": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _l, _vp],
    "pn2_sa_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _l, _vp],
    "pn2_fp_workspace_bytes": [_vp, _vp],
    "pn2_fp_forward": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _l, _vp],
    "pn2_fp_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _l, _vp],
    "pn2_fill_f32": [_l, _f, _vp, _vp],
    "pn2_box_sample": [_i, _l, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, ctypes.c_double, ctypes.c_double,
                       ctypes.c_double, _ull, _vp, _vp, _vp, _vp, _vp, _vp],
    "pn2_box_sample_key": [_ull, _i, _l],
    "pn2_adam_step": [_l, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _i, _f, _vp],
    "pn2_confusion_from_logits": [_l, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "pn2_confusion_from_labels": [_l, _i, _vp, _vp, _vp, _vp, _vp],
}
_RESTYPE = {"pn2_strerror": ctypes.c_char_p, "pn2_last_cuda_error": ctypes.c_char_p,
            "pn2_ball_threshold": ctypes.c_float, "pn2_linear_workspace_bytes": ctypes.c_long,
            "pn2_linear_image_bytes": ctypes.c_long, "pn2_box_sample_key": ctypes.c_uint,
            "pn2_sa_workspace_bytes": ctypes.c_long, "pn2_fp_workspace_bytes": ctypes.c_long,
            "pn2_ball_grid_workspace_bytes": ctypes.c_long}

_lib = None
launches = 0  # number of native entry-point calls made (bench.py reports it)
profile = None  # list of (name, start_event, end_event) when bench.py instruments a pass


class Pn2Error(RuntimeError):
    pass


def lib():
    """Load the shared library; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Pn2Error(
                "libpn2_b200.so is missing at %s -- build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` (there is no CPU fallback)"
                % LIB_PATH)
        _lib = ctypes.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(_lib, name)  # AttributeError if the ABI lost a symbol
            fn.argtypes = args
            fn.restype = _RESTYPE.get(name, ctypes.c_int)
    return _lib


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t, dtype=None, allow_none=False):
    """Raw device address of a contiguous CUDA tensor (None -> NULL when allowed)."""
    if t is None:
        if allow_none:
            return None
        raise Pn2Error("required tensor is None")
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise Pn2Error("pn2 ops need CUDA tensors (no CPU fallback); got %r" % (type(t),))
    if not t.is_contiguous():
        raise Pn2Error("pn2 ops need contiguous tensors")
    if dtype is not None and t.dtype != dtype:
        raise Pn2Error("expected dtype %s, got %s" % (dtype, t.dtype))
    return ctypes.c_void_p(t.data_ptr())


def ptr_rows(t, dtype=None):
    """(address, row pitch in elements) of a 2-D CUDA tensor whose rows are dense but may be padded
    (stride(1) == 1, stride(0) >= shape[1]), e.g. a column slice of a wider buffer."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dim() != 2:
        raise Pn2Error("pn2 ops need 2-D CUDA tensors here; got %r" % (type(t),))
    if t.shape[1] > 1 and t.stride(1) != 1 or t.stride(0) < t.shape[1]:
        raise Pn2Error("rows must be dense (unit column stride)")
    if dtype is not None and t.dtype != dtype:
        raise Pn2Error("expected dtype %s, got %s" % (dtype, t.dtype))
    return ctypes.c_void_p(t.data_ptr()), int(t.stride(0))


def call(name, *args):
    """Invoke an entry point on the current stream; map status codes to exceptions."""
    global launches
    if profile is not None:  # bench.py's instrumented pass: CUDA events around every call
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(lib(), name)(*args, stream())
        e1.record()
        profile.append((name, e0, e1, args[:3] if name in ("pn2_linear_fwd", "pn2_linear_fwd_bn", "pn2_linear_dgrad", "pn2_linear_wgrad") else None))
    else:
        rc = getattr(lib(), name)(*args, stream())
    launches += 1
    if rc != PN2_OK:
        msg = lib().pn2_strerror(rc).decode()
        if rc == PN2_EINVAL:
            raise ValueError("%s: %s" % (name, msg))
        detail = lib().pn2_last_cuda_error().decode()
        raise Pn2Error("%s: %s %s" % (name, msg, detail))
    return rc


F32, I32, F64 = torch.float32, torch.int32, torch.float64
