"""CPU restatement of nnU-Net v1's region-based inference (nnUNetTrainerV2BraTSRegions), marked [U] like
oracle/nnunet_oracle.py: recalled from upstream v1.7.x, not diffed against it (the fork is not installed).  It reuses that
module's Generic_UNet and tiled predictor unchanged and adds only what region-based models do differently:

  * [U:training/network_training/competitions_with_custom_Trainers/BraTS2020/nnUNetTrainerV2BraTSRegions.py]
    regions = get_brats_regions(), regions_class_order = (1, 2, 3), num_classes = len(regions) network outputs,
    network.inference_apply_nonlin = sigmoid (one per output, not a softmax over them).
  * [U:network_architecture/neural_network.py::_internal_predict_3D_3Dconv_tiled] with regions_class_order:
        seg = np.zeros(predicted_segmentation.shape[1:], dtype=np.float32)
        for i, c in enumerate(regions_class_order):
            seg[class_probabilities[i] > 0.5] = c
    (later regions overwrite earlier ones; exactly 0.5 and NaN are outside; the returned seg is float32).  Without it a
    sigmoid network still gets argmax(0).
  * [U:inference/segmentation_export.py::save_segmentation_nifti_from_softmax(region_class_order=...)]: the same rule on
    the probabilities resampled back to the cropped grid, then pasted back.

The sigmoid is applied by the oracle's own mirror_and_predict through net.inference_apply_nonlin; the tiled overlap-add
(`*=` on the tile, `+=` on the host) is the oracle's, in fp32.
"""
import numpy as np
import torch

import oracle as O

BRATS_REGIONS = {"whole tumor": (1, 2, 3), "tumor core": (2, 3), "enhancing tumor": (3,)}
BRATS_REGIONS_CLASS_ORDER = (1, 2, 3)


def region_labels(probs, regions_class_order):
    """Upstream's loop, as written there: probs [R, ...] -> float32 labels."""
    seg = np.zeros(probs.shape[1:], dtype=np.float32)
    for i, c in enumerate(regions_class_order):
        seg[probs[i] > 0.5] = c
    return seg


def build_region_network(plans, model_index=0, num_regions=3):
    """build_benchmark_network's seeded random init with num_regions sigmoid outputs (plans['num_classes'] is ignored: a
    region model's label count is not its output count)."""
    net = O.build_benchmark_network(model_index, dict(plans, num_classes=num_regions - 1))
    net.inference_apply_nonlin = torch.sigmoid
    return net


def predict_3D(net, x, do_mirroring, mirror_axes=(0, 1, 2), step_size=0.5, patch_size=None, regions_class_order=None,
               use_gaussian=True):
    """[U::SegmentationNetwork.predict_3D], tiled branch, for a sigmoid network: (seg, probabilities).  seg is the region
    rule (float32) with regions_class_order, argmax(0) without."""
    agg, nb = O.predict_3D_tiled(net, x, step_size, do_mirroring, mirror_axes, patch_size, use_gaussian, return_buffers=True)
    probs = agg / nb
    if regions_class_order is None:
        return probs.argmax(0), probs
    return region_labels(probs, regions_class_order), probs


class OracleRegionTrainer(O.OracleTrainer):
    """OracleTrainer with the region trainer's constants: sigmoid outputs and regions_class_order."""

    regions = BRATS_REGIONS
    regions_class_order = BRATS_REGIONS_CLASS_ORDER

    def __init__(self, plans, network):
        super().__init__(plans, network)
        self.num_classes = len(self.regions)
        assert network.num_classes == self.num_classes and network.inference_apply_nonlin is torch.sigmoid

    def predict_preprocessed_data_return_seg_and_softmax(self, data, do_mirroring=True, mirror_axes=None, step_size=0.5,
                                                         use_gaussian=True):
        if do_mirroring and mirror_axes is None:
            mirror_axes = self.data_aug_params["mirror_axes"]
        self.network.eval()
        with torch.no_grad():
            return predict_3D(self.network, data, do_mirroring, mirror_axes or (), step_size,
                              tuple(int(i) for i in self.patch_size), self.regions_class_order, use_gaussian)
