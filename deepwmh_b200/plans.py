"""`plans`-shaped dicts (the keys nnUNetTrainerV2.process_plans reads from plans.pkl, SURVEY.md A6)."""
from __future__ import annotations

from typing import Dict

import numpy as np


def benchmark_plans(patch_size=(128, 128, 128), num_pool: int = 5, base_num_features: int = 32,
                    num_modalities: int = 1, num_classes: int = 2) -> Dict:
    """The canonical 3d_fullres instance BASELINE.json is quoted on (SURVEY.md section 8d):
    1 modality, 2 classes, 5 stride-2 poolings, 3x3x3 kernels, patch 128^3.  num_classes counts the background."""
    return {
        "num_modalities": num_modalities, "num_classes": num_classes - 1,
        "base_num_features": base_num_features,
        "transpose_forward": [0, 1, 2], "transpose_backward": [0, 1, 2],
        "normalization_schemes": {m: "nonCT" for m in range(num_modalities)},
        "use_mask_for_norm": {m: True for m in range(num_modalities)},
        "plans_per_stage": {0: {
            "patch_size": np.array(patch_size),
            "pool_op_kernel_sizes": [[2, 2, 2]] * num_pool,
            "conv_kernel_sizes": [[3, 3, 3]] * (num_pool + 1),
            "current_spacing": np.array([1.0, 1.0, 1.0]),
            "batch_size": 2,
        }},
    }
