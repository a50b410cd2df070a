"""N4 bias-field correction on the GPU (dwmh_n4, csrc/n4.cu): the `N4BiasFieldCorrection -d 3 -c [50x50x50x50,0.0] -s 2`
step of DeepWMH_predict (deepwmh/main/predict.py:117-126) without the ANTs binary.  The algorithm and the points where it
may differ from ANTs are in DESIGN.md ("N4 bias-field correction").  There is no CPU path."""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np

from . import _lib

MAX_LEVELS = 8


def n4_bias_field_correction(volume, shrink_factor: int = 2, iterations: Sequence[int] = (50, 50, 50, 50), device: int = 0,
                             return_log_field: bool = False):
    """N4 of one [X][Y][Z] volume: returns volume / exp(B) (and B, the log bias field, with return_log_field) as float32.

    `volume` is a numpy array (computed on cuda:`device`, returned as numpy) or a CUDA tensor (computed on its own device,
    returned there).  `iterations` gives the iterations of each fitting level (the B-spline mesh doubles per level, at most
    8 levels).  Voxels <= 0 take no part in the fit and come back as volume / exp(B)."""
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("N4 bias-field correction runs on the GPU only (dwmh_n4) and no CUDA device is available")
    iters = [int(v) for v in iterations]
    if not 1 <= len(iters) <= MAX_LEVELS:
        raise ValueError("iterations: 1 to %d levels, got %d" % (MAX_LEVELS, len(iters)))
    is_numpy = not isinstance(volume, torch.Tensor)
    if is_numpy:
        vol = torch.from_numpy(np.ascontiguousarray(volume, dtype=np.float32)).to(torch.device("cuda", int(device)))
    else:
        if not volume.is_cuda:
            raise ValueError("a torch tensor input must be on a CUDA device")
        vol = volume.to(torch.float32).contiguous()
    if vol.dim() != 3:
        raise ValueError("expected one 3-D volume [X][Y][Z], got shape %s" % (tuple(vol.shape),))
    lib = _lib.load()
    X, Y, Z = (int(v) for v in vol.shape)
    nbytes = C.c_int64()
    _lib.check(lib.dwmh_n4_workspace(X, Y, Z, int(shrink_factor), len(iters), C.byref(nbytes)))
    it = (C.c_int32 * len(iters))(*iters)
    with torch.cuda.device(vol.device):
        ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=vol.device)
        out = torch.empty_like(vol)
        field = torch.empty_like(vol) if return_log_field else None
        _lib.check(lib.dwmh_n4(vol.device.index, _lib.ptr(vol), X, Y, Z, int(shrink_factor), len(iters), it, _lib.ptr(out),
                               _lib.ptr(field), _lib.ptr(ws), _lib.stream(vol.device)))
    if is_numpy:
        out = out.cpu().numpy()
        field = field.cpu().numpy() if field is not None else None
    return (out, field) if return_log_field else out
