"""ctypes binding of libdeepwmh_b200.so (include/deepwmh_b200.h).  Fails loudly: there is no CPU
or PyTorch fallback for any of these entry points."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

DWMH_MAX_POOL = 7
DWMH_MAX_IN_CHANNELS = 4
DWMH_MAX_CLASSES = 8


class NetDesc(C.Structure):
    _fields_ = [
        ("in_channels", C.c_int32), ("num_classes", C.c_int32), ("base_num_features", C.c_int32),
        ("max_num_features", C.c_int32), ("num_pool", C.c_int32), ("patch_size", C.c_int32 * 3),
        ("pool_op_kernel_sizes", (C.c_int32 * 3) * DWMH_MAX_POOL),
        ("conv_kernel_sizes", (C.c_int32 * 3) * (DWMH_MAX_POOL + 1)),
        ("act_dtype", C.c_int32), ("max_batch", C.c_int32), ("struct_size", C.c_int32),
    ]


# every symbol include/deepwmh_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "dwmh_last_error": (C.c_char_p, []),
    "dwmh_version": (C.c_int, []),
    "dwmh_create": (C.c_int, [C.POINTER(_P), C.c_int, C.POINTER(NetDesc)]),
    "dwmh_destroy": (C.c_int, [_P]),
    "dwmh_create_like": (C.c_int, [C.POINTER(_P), _P]),
    "dwmh_set_weight": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), C.c_int32]),
    "dwmh_commit_weights": (C.c_int, [_P]),
    "dwmh_zscore": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.POINTER(C.c_double), _P]),
    "dwmh_compute_steps": (C.c_int, [C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_double, C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]),
    "dwmh_gaussian_map": (C.c_int, [C.POINTER(C.c_int32), C.c_double, _P]),
    "dwmh_set_importance_map": (C.c_int, [_P, _P]),
    "dwmh_predict_3d": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32, C.c_int32, C.c_int32,
                                  _P, _P, C.c_int32, C.c_int32, _P]),
    "dwmh_weight_map": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32, _P, _P]),
    "dwmh_finalize": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P]),
    "dwmh_axpy": (C.c_int, [_P, _P, _P, C.c_float, C.c_int64, _P]),
    "dwmh_argmax": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int64, _P]),
    "dwmh_ensemble_masked_add": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P]),
    "dwmh_ensemble_refine": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int64, _P]),
    "dwmh_remove_sparks": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "dwmh_keep_largest_components": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_double, C.c_double, _P]),
    "dwmh_s1_zscore": (C.c_int, [C.c_int32, _P, _P, C.c_int64, C.c_int32, _P, C.POINTER(C.c_double), _P]),
    "dwmh_s1_zscore_batch": (C.c_int, [C.c_int32, C.POINTER(_P), C.c_int32, _P, C.c_int64, C.c_int32, _P, _P]),
    "dwmh_s1_local_mean_align_workspace": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int64)]),
    "dwmh_s1_local_mean_align": (C.c_int, [C.c_int32, _P, C.POINTER(_P), C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32,
                                           C.POINTER(C.c_int32), _P, _P, _P]),
    "dwmh_s1_mean_std_grid_workspace": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "dwmh_s1_mean_std_grid": (C.c_int, [C.c_int32, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), _P, _P, _P, _P]),
    "dwmh_s1_align_local_mean": (C.c_int, [C.c_int32, _P, _P, _P, C.c_int64, _P]),
    "dwmh_s1_group_nll": (C.c_int, [C.c_int32, _P, C.POINTER(_P), C.c_int32, C.c_double, C.c_int32, _P, _P, _P, _P, C.c_int64, _P]),
    "dwmh_s1_group_nll_masked": (C.c_int, [C.c_int32, _P, C.POINTER(_P), C.POINTER(_P), C.c_int32, C.c_double, C.c_int32, _P, _P, _P, _P,
                                           C.c_int64, _P]),
    "dwmh_s1_median_filter": (C.c_int, [C.c_int32, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), _P]),
    "dwmh_s1_component_filtering_workspace": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int64)]),
    "dwmh_s1_component_filtering": (C.c_int, [C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_double), _P, _P, _P]),
    "dwmh_s1_minmax": (C.c_int, [C.c_int32, _P, _P, C.c_int64, _P, C.POINTER(C.c_float), _P]),
    "dwmh_s1_histogram": (C.c_int, [C.c_int32, _P, _P, C.c_int64, C.c_int32, C.c_float, _P, C.c_int32, _P, _P]),
    "dwmh_s1_threshold_mask": (C.c_int, [C.c_int32, _P, C.c_float, _P, _P, C.c_int64, _P]),
    "dwmh_s1_masked_sums": (C.c_int, [C.c_int32, C.POINTER(_P), C.c_int32, _P, C.c_int64, C.c_int32, _P, C.POINTER(C.c_double), _P]),
    "dwmh_s1_label_vote": (C.c_int, [C.c_int32, C.POINTER(_P), C.c_int32, C.c_int32, _P, _P, C.c_int64, _P]),
    "dwmh_s1_apply_priors": (C.c_int, [C.c_int32, _P, _P, _P, _P, C.c_int32, C.c_int64, _P]),
    "dwmh_resample_workspace": (C.c_int, [C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.POINTER(C.c_int64)]),
    "dwmh_resample": (C.c_int, [C.c_int32, _P, C.POINTER(C.c_int32), _P, C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "dwmh_n4_workspace": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int64)]),
    "dwmh_n4": (C.c_int, [C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), _P, _P, _P, _P]),
    "dwmh_predict_volume_host": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32,
                                           C.c_int32, C.c_int32, _P, _P, _P]),
    "dwmh_predict_volume_host_masked": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32,
                                                  C.c_int32, C.c_int32, _P, _P, _P]),
    "dwmh_forward_patches": (C.c_int, [_P, _P, C.c_int32, _P, _P]),
    "dwmh_debug_layer_output": (C.c_int, [_P, C.c_int32, _P, C.c_int64, C.POINTER(C.c_int32), _P]),
    "dwmh_num_layers": (C.c_int, [_P]),
    "dwmh_layer_kernel_kind": (C.c_int, [_P, C.c_int32]),
    "dwmh_layer_norm_on_load": (C.c_int, [_P, C.c_int32]),
    "dwmh_set_force_generic": (C.c_int, [_P, C.c_int32]),
    "dwmh_get_counters": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "dwmh_set_stage_timing": (C.c_int, [_P, C.c_int32]),
    "dwmh_get_stage_timing": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "dwmh_get_kernel_timing": (C.c_int, [_P, C.POINTER(C.c_double)]),
}

_lib = None


class DwmhError(RuntimeError):
    pass


def lib_path() -> str:
    """The in-tree library; DWMH_LIB_PATH selects another build of it (A/B timing of two kernel versions on one box)."""
    return os.environ.get("DWMH_LIB_PATH") or _build.LIB_PATH


def load(build_if_missing: bool = True) -> C.CDLL:
    """dlopen the in-tree library (building it with nvcc first if it is absent)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise DwmhError(f"{path} is missing; run `python -m deepwmh_b200.build`")
        _build.build()
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        msg = load().dwmh_last_error()
        raise DwmhError(msg.decode() if msg else f"libdeepwmh_b200 error {rc}")


def compute_steps(patch, image, step_size):
    """_compute_steps_for_sliding_window through the C ABI (host only, no GPU needed)."""
    lib = load()
    p = (C.c_int32 * 3)(*[int(v) for v in patch])
    im = (C.c_int32 * 3)(*[int(v) for v in image])
    mx = 4096
    bufs = [(C.c_int32 * mx)() for _ in range(3)]
    cnt = (C.c_int32 * 3)()
    check(lib.dwmh_compute_steps(p, im, float(step_size), bufs[0], bufs[1], bufs[2], mx, cnt))
    return [[int(bufs[a][i]) for i in range(cnt[a])] for a in range(3)]


def gaussian_map(patch, sigma_scale=1.0 / 8) -> np.ndarray:
    """_get_gaussian closed form through the C ABI (host only)."""
    lib = load()
    p = (C.c_int32 * 3)(*[int(v) for v in patch])
    out = np.empty(tuple(int(v) for v in patch), dtype=np.float32)
    check(lib.dwmh_gaussian_map(p, float(sigma_scale), out.ctypes.data_as(C.c_void_p)))
    return out
