"""ctypes binding of ``libawb.so`` (C-ABI declared in ``include/awb.h``).

There is no CPU fallback: importing a kernel-backed symbol without the built
library raises ``AwbLibraryError`` (run ``python -c "import __graft_entry__ as g; g.build()"``).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AWB_LIB_PATH") or os.path.join(_HERE, "csrc", "libawb.so")   # override: A/B builds

AWB_KIND_ICNN, AWB_KIND_FLOW_ICNN, AWB_KIND_STAR, AWB_KIND_DIFFEO_ICNN = 0, 1, 2, 3
AWB_PREC_FP32, AWB_PREC_F16 = 0, 1
AWB_GRID_EXPLICIT, AWB_GRID_LINSPACE, AWB_GRID_INDEX = 0, 1, 2
AWB_WS_INFERENCE, AWB_WS_TRAINING, AWB_WS_FIT_STEP, AWB_WS_DEFORMATION, AWB_WS_SECOND_ORDER = 0, 1, 2, 3, 4
AWB_FWD_EXACT, AWB_FWD_EXACT_TRAINING, AWB_FWD_TC, AWB_FWD_TC_TRAINING = 0, 1, 2, 3
AWB_LOSS_SE_SIGMOID, AWB_LOSS_BCE_LOGITS = 0, 1
AWB_CLS_UNARY_LT_HALF, AWB_CLS_NOT_ONE = 0, 1
AWB_OPT_ADAM, AWB_OPT_ADAMAX = 0, 1
AWB_MAX_GROUPS = 4
AWB_FIT_REUSE_PACKED = 1


class AwbLibraryError(RuntimeError):
    pass


class AwbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libawb status {code}: {msg}")
        self.code = code


class Desc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("C", C.c_int32), ("h", C.c_int32), ("L", C.c_int32),
                ("F", C.c_int32), ("m", C.c_int32), ("flow_tanh", C.c_int32),
                ("n_objects", C.c_int32), ("precision", C.c_int32)]


class GridSpec(C.Structure):
    _fields_ = [("mode", C.c_int32), ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("t0", C.c_float), ("t_step", C.c_float), ("grid", C.c_void_p)]


class LossSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("cls_rule", C.c_int32), ("coef_fg", C.c_float), ("coef_bg", C.c_float),
                ("weight", C.c_void_p), ("ignore_enabled", C.c_int32), ("ignore_value", C.c_float)]


class OptHyper(C.Structure):
    _fields_ = [("kind", C.c_int32), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float * AWB_MAX_GROUPS),
                ("plateau_enabled", C.c_int32), ("patience", C.c_int32),
                ("factor", C.c_float), ("threshold", C.c_float), ("min_lr", C.c_float),
                ("plateau_eps", C.c_float), ("active_groups", C.c_int32)]


class OptScalars(C.Structure):
    _fields_ = [("step", C.c_int32), ("num_bad", C.c_int32), ("nonfinite", C.c_int32), ("pad", C.c_int32),
                ("lr", C.c_double * AWB_MAX_GROUPS), ("best", C.c_double),
                ("last_loss", C.c_float), ("pad2", C.c_float)]


# every symbol include/awb.h declares: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("awb_version", C.c_char_p, []),
    ("awb_last_error", C.c_char_p, []),
    ("awb_prior_create", C.c_int, [C.POINTER(Desc), C.POINTER(_P)]),
    ("awb_prior_destroy", C.c_int, [_P]),
    ("awb_prior_param_count", C.c_int64, [_P]),
    ("awb_prior_workspace_bytes", C.c_int64, [_P, C.c_int64, C.c_int32]),
    ("awb_opt_state_bytes", C.c_int64, [_P]),
    ("awb_prior_set_flow_consts", C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_float,
                                            C.c_float, C.POINTER(C.c_uint8)]),
    ("awb_prior_set_flow_output_scale", C.c_int, [_P, C.c_float]),
    ("awb_prior_set_flow_eval", C.c_int, [_P, C.c_int32]),
    ("awb_prior_forward", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, _P, C.c_int32, _P, C.c_size_t, _P]),
    ("awb_prior_flow_inverse", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, _P]),
    ("awb_prior_backward", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, _P, _P, _P, C.c_size_t, _P]),
    ("awb_prior_grid_grad_backward", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, _P, _P, _P, _P, C.c_size_t, _P]),
    ("awb_prior_deformation", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, C.c_int32, _P, C.c_size_t, _P]),
    ("awb_prior_deformation_backward", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, _P, _P, _P, C.c_size_t, _P]),
    ("awb_prior_inverse", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, C.c_int32, _P, C.c_size_t, _P]),
    ("awb_prior_inverse_backward", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, _P, _P, _P, C.c_size_t, _P]),
    ("awb_prior_fit_step", C.c_int, [_P, _P, _P, C.POINTER(GridSpec), _P, C.POINTER(LossSpec),
                                     C.POINTER(OptHyper), _P, _P, C.c_size_t, C.c_int32, _P]),
    ("awb_prior_fit_steps", C.c_int, [_P, _P, _P, C.POINTER(GridSpec), C.POINTER(_P), C.c_int32, C.c_int32, C.c_int32,
                                      C.POINTER(LossSpec), C.POINTER(OptHyper), _P, _P, C.c_size_t, C.c_int32, _P]),
    ("awb_prior_fit_host_frames", C.c_int, [_P, _P, _P, C.POINTER(GridSpec), C.POINTER(_P), C.c_int32, C.c_int32,
                                            C.POINTER(LossSpec), C.POINTER(OptHyper), _P, _P, _P, C.c_size_t,
                                            C.c_int32, _P]),
    ("awb_prior_grad_row_floats", C.c_int64, [_P]),
    ("awb_prior_slice_grads", C.c_int, [_P, _P, C.POINTER(GridSpec), C.c_int64, C.c_int64, _P, C.POINTER(LossSpec), _P,
                                        _P, C.c_size_t, C.c_int32, _P]),
    ("awb_prior_rows_opt_step", C.c_int, [_P, _P, _P, _P, C.c_int32, C.POINTER(OptHyper), _P, _P, C.c_size_t, _P]),
    ("awb_flow_identity_step", C.c_int, [_P, _P, _P, C.POINTER(GridSpec), C.POINTER(OptHyper), _P, _P,
                                         C.c_size_t, _P]),
    ("awb_optim_step", C.c_int, [_P, _P, _P, _P, C.POINTER(OptHyper), _P]),
    ("awb_prior_enforce_convexity", C.c_int, [_P, _P, _P]),
    ("awb_opt_state_init", C.c_int, [_P, _P, C.POINTER(C.c_double), _P]),
    ("awb_star_forward", C.c_int, [_P, _P, _P, C.c_int64, _P, _P]),
    ("awb_star_workspace_bytes", C.c_int64, [_P, C.c_int64]),
    ("awb_star_fit_step", C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.POINTER(LossSpec), C.POINTER(OptHyper), _P, _P,
                                    C.c_size_t, _P]),
    ("awb_star_backward_workspace_bytes", C.c_int64, [_P, C.c_int64]),
    ("awb_star_backward", C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, _P, C.c_size_t, _P]),
    ("awb_opt_set_lr", C.c_int, [_P, _P, C.POINTER(C.c_double), _P]),
    ("awb_opt_plateau_step", C.c_int, [_P, _P, _P, C.c_int32, C.POINTER(OptHyper), _P]),
    ("awb_opt_read_scalars", C.c_int, [_P, _P, C.c_int32, C.POINTER(OptScalars), _P]),
    ("awb_prior_actnorm_init", C.c_int, [_P, _P, C.POINTER(GridSpec), _P, C.c_size_t, _P]),
    ("awb_mask_iou_counts", C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P]),
    ("awb_target_counts", C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, _P]),
    ("awb_target_counts_ignore", C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P]),
    ("awb_image_process", C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    ("awb_image_edge_map", C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P]),
    ("awb_debug_umma_probe", C.c_int, [_P, C.c_int32, _P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                       C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), _P]),
    ("awb_debug_tc_trace_read", C.c_int, [C.POINTER(C.c_ulonglong), C.c_int32]),
    ("awb_profile_enable", C.c_int, [C.c_int32]),
    ("awb_profile_classes", C.c_int, []),
    ("awb_profile_class_name", C.c_char_p, [C.c_int32]),
    ("awb_profile_read", C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    ("awb_launch_count", C.c_longlong, []),
]

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load libawb.so (once) and type every exported symbol.  Raises loudly when absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AwbLibraryError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built "
            "(python -c 'import __graft_entry__ as g; g.build()').  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)     # AttributeError if the header and the library disagree
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise AwbError(rc, load().awb_last_error().decode())


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda() -> None:
    import torch
    if not torch.cuda.is_available():
        raise AwbLibraryError("awesome_b200 needs a CUDA device (sm_100a); there is no CPU fallback.")
