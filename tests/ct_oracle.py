"""CPU restatement of what nnU-Net v1 does for CT models and the cascade, marked [U] like oracle/nnunet_oracle.py: recalled
from upstream v1.7.x, not diffed against it (nnunet is not installed).  It adds to oracle/resample_oracle.py only what these
models do differently:

  * [U:preprocessing/preprocessing.py::GenericPreprocessor.resample_and_normalize] per modality c, after the resample, with
    ip = plans['dataset_properties']['intensityproperties'][c]:
        "CT":     data[c] = np.clip(data[c], ip['percentile_00_5'], ip['percentile_99_5'])
                  data[c] = (data[c] - ip['mean']) / ip['sd']
        "CT2":    mask = (data[c] > lb) & (data[c] < ub); data[c] = np.clip(data[c], lb, ub)
                  mn = data[c][mask].mean(); sd = data[c][mask].std(); data[c] = (data[c] - mn) / sd
        "noNorm": nothing
    then, if use_nonzero_mask[c]: data[c][seg[-1] < 0] = 0.  data is float32 and the constants are python floats, which
    numpy 1.x applies in float32: ct_normalize rounds them to float32 and computes in float32.  ct2_normalize takes mn / sd in
    float64 (the device's accumulation) where numpy uses its float32 pairwise sums: CT2 is held to a tolerance.
  * [U:inference/predict.py::preprocess_save_to_queue] a 3d_cascade_fullres case: seg_prev (the previous stage's labels in
    the raw image's geometry) -> transpose(transpose_forward) -> resize_segmentation(seg_prev, d.shape[1:], order=1) ->
    to_one_hot(.., classes 1 .. C-1) appended after the normalised modalities.  The map is the UNCROPPED one, resized onto
    the cropped, resampled grid.
  * [U:training/network_training/nnUNetTrainerV2_CascadeFullRes.py] that network has num_modalities + num_classes - 1
    inputs and the largest stage; 3d_lowres is the smallest stage.
"""
import numpy as np

import oracle as O
import oracle.resample_oracle as R
from deepwmh_b200 import preprocess


def ct_normalize(x, lb, ub, mean, sd, seg=None):
    """"CT" in float32 (seg: crop mask, zeroed where < 0, or None)."""
    f = np.float32
    y = np.clip(np.asarray(x, np.float32), f(lb), f(ub))
    y = (y - f(mean)) / f(sd)
    if seg is not None:
        y[np.asarray(seg) < 0] = 0
    return y.astype(np.float32)


def ct2_stats(x, lb, ub):
    """CT2's (mean, population std, count) of the values strictly inside (lb, ub), in float64."""
    x = np.asarray(x, np.float32)
    v = x[(x > np.float32(lb)) & (x < np.float32(ub))].astype(np.float64)
    return float(v.mean()), float(v.std()), int(v.size)


def ct2_normalize(x, lb, ub, seg=None):
    """"CT2" with float64 statistics applied in float32."""
    mn, sd, _ = ct2_stats(x, lb, ub)
    return ct_normalize(x, lb, ub, mn, sd, seg)


def to_one_hot(seg, num_classes):
    """[U:utilities/one_hot_encoding.py::to_one_hot] over classes 1 .. num_classes-1, float32."""
    return np.stack([(seg == c) for c in range(1, num_classes)]).astype(np.float32)


def cascade_channels(seg_prev, shape, num_classes):
    """resize_segmentation(seg_prev, shape, order=1) one-hot over classes 1 .. num_classes-1."""
    return to_one_hot(R.resize_segmentation(np.asarray(seg_prev), shape, order=1), num_classes)


def stage_plans(plans, stage):
    """The plans with only plans_per_stage[stage] (the oracle's network and trainer take the largest stage)."""
    return dict(plans, plans_per_stage={stage: plans["plans_per_stage"][stage]})


def preprocess_case(plans, data, spacing, stage=None, seg_prev=None):
    """crop_to_nonzero -> resample to the stage's spacing -> per-modality scheme -> (cascade) one-hot previous stage.
    data float32 [M, z, y, x] with transpose_forward = identity; spacing (z, y, x).  Returns (d float32, crop bbox, cropped
    shape, target spacing)."""
    stage = max(plans["plans_per_stage"]) if stage is None else stage
    target = np.array(plans["plans_per_stage"][stage]["current_spacing"], dtype=np.float64)
    cropped, seg, bbox = preprocess.crop_to_nonzero(data)
    d, s = R.resample_patient(cropped, seg, np.array(spacing, dtype=np.float64), target, 3, 1, force_separate_z=None)
    s = s.copy()
    s[s < -1] = 0
    out = d.astype(np.float32)
    ips = plans.get("dataset_properties", {}).get("intensityproperties", {})
    for c in range(out.shape[0]):
        scheme = plans["normalization_schemes"][c]
        mask = s[-1] if plans["use_mask_for_norm"][c] else None
        if scheme == "CT":
            ip = ips[c]
            out[c] = ct_normalize(out[c], ip["percentile_00_5"], ip["percentile_99_5"], ip["mean"], ip["sd"], mask)
        elif scheme == "CT2":
            ip = ips[c]
            out[c] = ct2_normalize(out[c], ip["percentile_00_5"], ip["percentile_99_5"], mask)
        elif scheme == "nonCT":
            out[c] = O.zscore_nnunet(out[c], s[-1], plans["use_mask_for_norm"][c])
    if seg_prev is not None:
        out = np.concatenate([out, cascade_channels(seg_prev, out.shape[1:], plans["num_classes"] + 1)])
    return out, bbox, cropped.shape[1:], target


def predict_case(plans, net, data, spacing, stage=None, seg_prev=None):
    """The whole oracle pipeline of one case -> (labels uint8 in the raw geometry, softmax resampled back to the crop)."""
    stage = max(plans["plans_per_stage"]) if stage is None else stage
    d, bbox, crop_shape, target = preprocess_case(plans, data, spacing, stage, seg_prev)
    sp = stage_plans(plans, stage)
    if seg_prev is not None:
        sp = dict(sp, num_modalities=d.shape[0])
    _, p = O.OracleTrainer(sp, net.float()).predict_preprocessed_data_return_seg_and_softmax(d)
    p = R.resample_softmax_back(p, crop_shape, np.array(spacing, dtype=np.float64), target)
    return preprocess.paste_back(p.argmax(0).astype(np.uint8), data.shape[1:], bbox), p
