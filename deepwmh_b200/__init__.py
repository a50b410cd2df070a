"""deepwmh_b200 -- B200-native drop-in for DeepWMH's nnU-Net 3d_fullres sliding-window inference.

Only what the hot path needs lives here: `csrc/` (hand-written sm_100a CUDA + the C ABI of
include/deepwmh_b200.h), the ctypes binding, and the host-side mirror of the nnU-Net predictor
surface (`nnUNetTrainerV2.predict_preprocessed_data_return_seg_and_softmax`,
`SegmentationNetwork.predict_3D`).  Importing the package never imports `oracle/`.
"""
from . import _lib  # noqa: F401
from .plans import benchmark_plans  # noqa: F401
from .predictor import (SegmentationNetwork, nnUNetTrainerV2, nnUNetTrainerV2BraTSRegions,  # noqa: F401
                        nnUNetTrainerV2CascadeFullRes, pad_nd_image)

__all__ = ["SegmentationNetwork", "nnUNetTrainerV2", "nnUNetTrainerV2BraTSRegions", "nnUNetTrainerV2CascadeFullRes", "benchmark_plans",
           "pad_nd_image"]
