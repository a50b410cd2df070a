"""File-level steps either side of the hot path (SURVEY.md section 8f-1/8f-2), host side.

Restates, for DeepWMH's single modality and for models with up to four, what nnU-Net v1 does around predict_3D:
  * crop_to_nonzero                      [U:preprocessing/cropping.py]      (scipy binary_fill_holes, as upstream)
  * paste-back export                    [U:inference/segmentation_export.py]
  * remove_3mm_sparks                    deepwmh/analysis/image_ops.py:325-367 (scipy.ndimage.label, as the reference)
  * spacing resample                     [U:preprocessing/preprocessing.py::resample_patient / resample_data_or_seg]: the
    shape / separate-z decisions here on the host, the spline arithmetic on the device (dwmh_resample, csrc/resample.cu)
  * preprocess_test_case / resample-back [U:GenericPreprocessor.preprocess_test_case,
                                          inference/segmentation_export.py::save_segmentation_nifti_from_softmax]
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
from scipy.ndimage import binary_fill_holes, label


def crop_to_nonzero(data: np.ndarray) -> Tuple[np.ndarray, np.ndarray, List[List[int]]]:
    """data [c, z, y, x] -> (cropped data, seg [1, z, y, x] with -1 outside the filled nonzero mask and 0 inside,
    bbox [[z0, z1], [y0, y1], [x0, x1]])."""
    assert data.ndim == 4
    mask = np.zeros(data.shape[1:], dtype=bool)
    for c in range(data.shape[0]):
        mask |= data[c] != 0
    mask = binary_fill_holes(mask)
    idx = np.where(mask)
    if idx[0].size == 0:
        bbox = [[0, s] for s in data.shape[1:]]
    else:
        bbox = [[int(idx[a].min()), int(idx[a].max()) + 1] for a in range(3)]
    sl = tuple(slice(b[0], b[1]) for b in bbox)
    cropped = data[(slice(None),) + sl]
    seg = np.where(mask[sl], 0, -1).astype(np.int8)[None]
    return np.ascontiguousarray(cropped), seg, bbox


RESAMPLING_SEPARATE_Z_ANISO_THRESHOLD = 3


def resampled_shape(shape: Sequence[int], original_spacing, target_spacing) -> np.ndarray:
    """[U:resample_patient] new_shape = round(original_spacing / target_spacing * shape) (numpy round: half to even)."""
    return np.round((np.array(original_spacing) / np.array(target_spacing)).astype(float) * np.array(shape)).astype(int)


def _lowres_axis(spacing) -> np.ndarray:
    return np.where(max(spacing) / np.array(spacing) == 1)[0]


def separate_z_rule(original_spacing, target_spacing, force_separate_z=None, threshold=RESAMPLING_SEPARATE_Z_ANISO_THRESHOLD):
    """[U:resample_patient] -> (do_separate_z, axis or None): separate z when max/min spacing > 3 of the original (else of
    the target) spacing, on the single axis carrying the largest spacing; two or three tied axes switch it off."""
    if force_separate_z is not None:
        do, axis = bool(force_separate_z), (_lowres_axis(original_spacing) if force_separate_z else None)
    elif np.max(original_spacing) / np.min(original_spacing) > threshold:
        do, axis = True, _lowres_axis(original_spacing)
    elif np.max(target_spacing) / np.min(target_spacing) > threshold:
        do, axis = True, _lowres_axis(target_spacing)
    else:
        do, axis = False, None
    if axis is not None and len(axis) != 1:
        do = False
    return do, (int(axis[0]) if (do and axis is not None) else None)


def resample_device(vol, new_shape, order: int, separate_axis: Optional[int] = None, out_mode: int = 0):
    """One fp32 CUDA volume [x, y, z] -> new_shape with skimage.transform.resize semantics (dwmh_resample).
    out_mode 1: int8 {-1, 0} crop-mask labels from the 0/1 indicator of label 0 (resize_segmentation, order 1)."""
    import ctypes as C

    import torch

    from . import _lib
    lib = _lib.load()
    assert vol.is_cuda and vol.dtype == torch.float32 and vol.dim() == 3
    vol = vol.contiguous()
    new_shape = tuple(int(v) for v in new_shape)
    ins = (C.c_int32 * 3)(*vol.shape)
    outs = (C.c_int32 * 3)(*new_shape)
    sep = -1 if separate_axis is None else int(separate_axis)
    nbytes = C.c_int64()
    _lib.check(lib.dwmh_resample_workspace(ins, int(order), sep, C.byref(nbytes)))
    with torch.cuda.device(vol.device):
        ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=vol.device)
        out = torch.empty(new_shape, dtype=torch.int8 if out_mode == 1 else torch.float32, device=vol.device)
        _lib.check(lib.dwmh_resample(vol.device.index, _lib.ptr(vol), ins, _lib.ptr(out), outs, int(order), sep, int(out_mode),
                                     _lib.ptr(ws), _lib.stream(vol.device)))
    return out


def resample_patient_device(data, seg, original_spacing, target_spacing, force_separate_z=None):
    """[U:resample_patient] as GenericPreprocessor.resample_and_normalize calls it (data order 3, seg order 1, order_z 0)
    on CUDA tensors: data fp32 [c, x, y, z], seg int8 [1, x, y, z] with labels {-1, 0} (or None)."""
    import torch
    shape = tuple(data.shape[1:])
    new_shape = tuple(int(v) for v in resampled_shape(shape, original_spacing, target_spacing))
    if new_shape == shape:
        return data, seg
    do_sep, axis = separate_z_rule(original_spacing, target_spacing, force_separate_z)
    axis = axis if do_sep else None
    d = torch.stack([resample_device(data[c], new_shape, 3, axis) for c in range(data.shape[0])])
    s = None
    if seg is not None:
        ind = (seg[0] == 0).to(torch.float32)
        s = resample_device(ind, new_shape, 1, axis, out_mode=1)[None]
    return d, s


def resample_softmax_back_device(softmax, shape_after_cropping, original_spacing, spacing_after_resampling, force_separate_z=None,
                                 interpolation_order: int = 1):
    """[U:save_segmentation_nifti_from_softmax] class probabilities [classes, x, y, z] (after transpose_backward) back to
    the cropped original grid: order 1, separate-z decided on the ORIGINAL spacing first, then on the resampled one."""
    import torch
    shape_after_cropping = tuple(int(v) for v in shape_after_cropping)
    if tuple(softmax.shape[1:]) == shape_after_cropping:
        return softmax
    do_sep, axis = separate_z_rule(original_spacing, spacing_after_resampling, force_separate_z)
    return torch.stack([resample_device(softmax[c].contiguous(), shape_after_cropping, interpolation_order, axis if do_sep else None)
                        for c in range(softmax.shape[0])])


def paste_back(seg_cropped: np.ndarray, original_shape: Sequence[int], bbox: List[List[int]]) -> np.ndarray:
    out = np.zeros(tuple(original_shape), dtype=np.uint8)
    out[tuple(slice(b[0], b[1]) for b in bbox)] = seg_cropped
    return out


def remove_sparks(mask: np.ndarray, min_volume: int = 3) -> np.ndarray:
    """Discard connected components (6-connectivity, scipy default) smaller than min_volume voxels."""
    m = (mask > 0.5).astype(np.int32)
    lab, n = label(m)
    if n == 0:
        return np.zeros_like(m)
    sizes = np.bincount(lab.ravel(), minlength=n + 1)
    keep = sizes >= min_volume
    keep[0] = False
    return keep[lab].astype(np.int32)


def remove_3mm_sparks(mask: np.ndarray, voxel_size: Sequence[float]) -> np.ndarray:
    """deepwmh/analysis/image_ops.py:346-367: components below 3 mm^3 (>= 2 voxels) are removed; for thick-slice
    data (anisotropy > 3) the limit is 3 voxels."""
    vs = [float(v) for v in voxel_size]
    if max(vs) / min(vs) > 3.0:
        return remove_sparks(mask, 3)
    mv = int(np.around(3.0 / (vs[0] * vs[1] * vs[2])))
    return remove_sparks(mask, max(mv, 2))


def read_modalities(input_files: Sequence[str]):
    """The M modality files of one case (`<case>_0000 ... <case>_000{M-1}`) -> (data fp32 [M, z, y, x] in SimpleITK axis order,
    header of the first file).  The files must agree in shape, spacing and orientation, as nnU-Net requires."""
    from . import nifti
    vols, hdr0 = [], None
    for i, f in enumerate(input_files):
        vol_xyz, hdr = nifti.read_nifti(f)
        if hdr0 is None:
            hdr0 = hdr
        else:
            if tuple(hdr["shape"]) != tuple(hdr0["shape"]):
                raise ValueError("modality %d (%s) has shape %s, modality 0 has %s" % (i, f, tuple(hdr["shape"]), tuple(hdr0["shape"])))
            if not np.allclose(hdr["spacing"], hdr0["spacing"], rtol=1e-5, atol=1e-6) or not np.allclose(hdr["srow"], hdr0["srow"], rtol=1e-5, atol=1e-5):
                raise ValueError("modality %d (%s) does not share the geometry (spacing / affine) of modality 0 (%s)" % (i, f, input_files[0]))
        vols.append(np.transpose(vol_xyz, (2, 1, 0)))
    return np.ascontiguousarray(np.stack(vols)).astype(np.float32), hdr0


NORMALIZATION_SCHEMES = ("nonCT", "CT", "CT2", "noNorm")


def normalization_schemes(plans: Dict) -> List[Tuple[str, Optional[Dict[str, float]]]]:
    """[U:GenericPreprocessor.resample_and_normalize] each modality's scheme and, for CT / CT2, its constants from
    plans['dataset_properties']['intensityproperties'][c] as floats.  Raises NotImplementedError for a scheme other than
    nonCT, CT, CT2 or noNorm and for a CT / CT2 modality whose plans lack one of the constants; ValueError for constants
    the CT kernels refuse (non-finite, lb > ub, sd <= 0).  Reads nothing but the plans."""
    M = int(plans.get("num_modalities", 1))
    schemes = plans.get("normalization_schemes") or {}
    props = (plans.get("dataset_properties") or {}).get("intensityproperties") or {}
    out = []
    for m in range(M):
        scheme = schemes.get(m, "nonCT")
        if scheme not in NORMALIZATION_SCHEMES:
            raise NotImplementedError("normalization scheme %r of modality %d: nnU-Net's %s are implemented"
                                      % (scheme, m, ", ".join(NORMALIZATION_SCHEMES)))
        if scheme not in ("CT", "CT2"):
            out.append((scheme, None))
            continue
        keys = ("percentile_00_5", "percentile_99_5") + (("mean", "sd") if scheme == "CT" else ())
        ip = props.get(m)
        missing = [k for k in keys if ip is None or k not in ip]
        if missing:
            raise NotImplementedError("normalization scheme %r of modality %d needs plans['dataset_properties']['intensityproperties'][%d]"
                                      "[%s]; these plans lack it" % (scheme, m, m, "], [".join(repr(k) for k in missing)))
        c = {k: float(ip[k]) for k in keys}
        with np.errstate(over="ignore"):
            f32 = {k: np.float32(v) for k, v in c.items()}
        if not all(np.isfinite(v) for v in f32.values()) or f32["percentile_00_5"] > f32["percentile_99_5"]:
            raise ValueError("intensityproperties[%d] of scheme %r: %s (finite in float32, percentile_00_5 <= percentile_99_5)"
                             % (m, scheme, c))
        if scheme == "CT" and not f32["sd"] > 0:
            raise ValueError("intensityproperties[%d]['sd'] = %r: the CT scheme divides by it" % (m, c["sd"]))
        out.append((scheme, c))
    return out


def ct_normalize_device(vol, seg, scheme: str, constants: Dict[str, float]):
    """nnU-Net's CT or CT2 scheme in place on one fp32 CUDA volume (dwmh_ct_normalize); seg: int8 crop mask (zeroed where
    < 0) or None.  Returns CT2's (mean, sd, mask count) -- which synchronises the stream -- and None for CT."""
    import ctypes as C

    import torch

    from . import _lib
    lib = _lib.load()
    assert vol.is_cuda and vol.dtype == torch.float32 and vol.is_contiguous()
    assert seg is None or (seg.dtype == torch.int8 and seg.is_contiguous() and seg.numel() == vol.numel())
    ct2 = scheme == "CT2"
    code = _lib.DWMH_NORM_CT2 if ct2 else _lib.DWMH_NORM_CT
    stats = (C.c_double * 3)() if ct2 else None
    with torch.cuda.device(vol.device):
        ws = torch.empty(_lib.DWMH_CT_WORKSPACE_BYTES, dtype=torch.uint8, device=vol.device) if ct2 else None
        _lib.check(lib.dwmh_ct_normalize(vol.device.index, _lib.ptr(vol), _lib.ptr(seg),
                                         vol.numel(), code, constants["percentile_00_5"], constants["percentile_99_5"],
                                         constants.get("mean", 0.0), constants.get("sd", 1.0), stats, _lib.ptr(ws),
                                         _lib.stream(vol.device)))
    return tuple(stats) if ct2 else None


def cascade_onehot_device(labels, out, num_classes: int):
    """The cascade's previous-stage channels (dwmh_cascade_onehot): uint8 CUDA labels [x, y, z] -> resize_segmentation(order
    1) onto out's grid -> one-hot over classes 1 .. num_classes-1 written into out, fp32 CUDA [num_classes-1, X, Y, Z]."""
    import ctypes as C

    import torch

    from . import _lib
    lib = _lib.load()
    assert labels.is_cuda and labels.dtype == torch.uint8 and labels.dim() == 3
    assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.dim() == 4 and out.shape[0] == num_classes - 1
    labels = labels.contiguous()
    ins = (C.c_int32 * 3)(*labels.shape)
    outs = (C.c_int32 * 3)(*out.shape[1:])
    with torch.cuda.device(out.device):
        _lib.check(lib.dwmh_cascade_onehot(out.device.index, _lib.ptr(labels), ins, _lib.ptr(out), outs, int(num_classes),
                                           _lib.stream(out.device)))
    return out


def read_prev_stage_labels(label_file: str, image_shape: Sequence[int], num_classes: int) -> np.ndarray:
    """[U:inference/predict.py::preprocess_save_to_queue] the previous stage's label map of a cascade case in SimpleITK
    axis order (z, y, x), uint8.  Its NIfTI shape must be image_shape (the first modality file's) and its values labels
    0 .. num_classes-1."""
    from . import nifti
    if not os.path.isfile(label_file):
        raise RuntimeError("the previous stage's segmentation %s does not exist" % label_file)
    lab, _ = nifti.read_nifti(label_file)
    if tuple(lab.shape) != tuple(image_shape):
        raise ValueError("the previous stage's segmentation %s has shape %s, the case's images %s"
                         % (label_file, tuple(lab.shape), tuple(image_shape)))
    bad = ~np.isin(lab, np.arange(num_classes))
    if bad.any():
        raise ValueError("the previous stage's segmentation %s holds values %s outside the labels 0 .. %d of the model"
                         % (label_file, ", ".join("%g" % v for v in np.unique(lab[bad])[:8]), num_classes - 1))
    return np.ascontiguousarray(np.transpose(lab, (2, 1, 0))).astype(np.uint8)


def preprocess_test_case(network, plans: Dict, input_files: Sequence[str], force_separate_z=None, stage=None,
                         segs_from_prev_stage: Optional[str] = None):
    """[U:GenericPreprocessor.preprocess_test_case] for M = plans['num_modalities'] modalities (`<case>_0000 ...`; DeepWMH: one
    FLAIR): read (SimpleITK axis order z, y, x) -> crop_to_nonzero (nonzero mask over all modalities, holes filled) ->
    transpose_forward -> NaN -> 0 -> resample every modality to the spacing of plans stage `stage` (default: the largest
    key; device) -> normalise every modality by its scheme with its own use_mask_for_norm (device): nonCT (z-score), CT, CT2
    or noNorm (normalization_schemes).  segs_from_prev_stage: a 3d_cascade_fullres case's previous-stage label file
    (read_prev_stage_labels): after transpose_forward, resize_segmentation(order 1) of the UNCROPPED map onto the cropped,
    resampled grid, one-hot over classes 1 .. C-1, appended after the M modalities without normalisation.  Returns (data
    fp32 CUDA [M (+ C-1), x, y, z], seg int8 CUDA [1, x, y, z], properties)."""
    import torch

    M = int(plans.get("num_modalities", 1))
    if len(input_files) != M:
        raise ValueError("the model takes %d modalities; got %d input files" % (M, len(input_files)))
    norm = normalization_schemes(plans)
    stage = max(plans["plans_per_stage"].keys()) if stage is None else stage
    num_classes = int(plans["num_classes"]) + 1
    data, hdr = read_modalities(input_files)
    prev = read_prev_stage_labels(segs_from_prev_stage, hdr["shape"], num_classes) if segs_from_prev_stage is not None else None
    target_spacing = np.array(plans["plans_per_stage"][stage]["current_spacing"], dtype=np.float64)
    tf = list(plans.get("transpose_forward", [0, 1, 2]))
    props = {"original_size_of_raw_data": np.array(data.shape[1:]), "original_spacing": np.array(hdr["spacing"][::-1], dtype=np.float64),
             "list_of_data_files": list(input_files), "seg_file": None, "nifti_header": hdr}
    cropped, seg, bbox = crop_to_nonzero(data)
    props["crop_bbox"] = bbox
    props["classes"] = np.array([-1, 0])
    props["size_after_cropping"] = cropped.shape[1:]
    cropped = np.ascontiguousarray(cropped.transpose([0] + [i + 1 for i in tf]))
    seg = np.ascontiguousarray(seg.transpose([0] + [i + 1 for i in tf]))
    cropped[np.isnan(cropped)] = 0
    original_spacing_transposed = props["original_spacing"][tf]
    mask_for_norm = plans.get("use_mask_for_norm", {0: False})
    use_mask = [bool(mask_for_norm[m]) for m in range(M)]
    case = os.path.basename(input_files[0])

    def normalize(v, mask, m):
        scheme, constants = norm[m]
        if scheme == "nonCT":
            network.normalize_(v, mask if use_mask[m] else None, 1 if use_mask[m] else 0, return_stats=False)
        elif scheme in ("CT", "CT2"):
            stats = ct_normalize_device(v, mask if use_mask[m] else None, scheme, constants)
            if stats is not None and stats[2] == 0:
                raise ValueError("%s, modality %d: no voxel lies strictly between the CT2 bounds %r and %r, so the scheme has no "
                                 "mean or standard deviation" % (case, m, constants["percentile_00_5"], constants["percentile_99_5"]))

    with torch.cuda.device(network.device):
        d = torch.from_numpy(cropped).to(network.device)
        sg = torch.from_numpy(seg).to(network.device)
        d, sg = resample_patient_device(d, sg, original_spacing_transposed, target_spacing, force_separate_z)
        props["size_after_resampling"] = tuple(d.shape[1:])
        props["spacing_after_resampling"] = target_spacing
        props["use_nonzero_mask_for_norm"] = {m: use_mask[m] for m in range(M)}
        if M == 1:
            v = d[0].contiguous()
            normalize(v, sg[0].contiguous(), 0)
            d = v[None]
        else:
            d = d.contiguous()
            mask = sg[0].contiguous()
            # each channel of d starts 16-byte aligned only if X*Y*Z % 4 == 0: normalise a padded copy otherwise
            chans = []
            for m in range(M):
                v = d[m].clone() if d[0].numel() % 4 else d[m]
                normalize(v, mask, m)
                chans.append(v)
            d = torch.stack(chans) if d[0].numel() % 4 else d
        if prev is not None:
            x = torch.empty((M + num_classes - 1,) + tuple(d.shape[1:]), dtype=torch.float32, device=network.device)
            x[:M] = d
            labels = torch.from_numpy(np.ascontiguousarray(prev.transpose(tf))).to(network.device)
            cascade_onehot_device(labels, x[M:], num_classes)
            d = x
    return d, sg, props


def save_segmentation_nifti_from_softmax(network, softmax, out_fname: str, properties: Dict, order: int = 1, force_separate_z=None,
                                         softmax_fname: Optional[str] = None, post3mm_fname: Optional[str] = None,
                                         for_which_classes=None, min_valid_object_sizes=None, region_class_order=None):
    """[U:inference/segmentation_export.py::save_segmentation_nifti_from_softmax]: softmax [classes, x, y, z] (ALREADY
    transposed back; CUDA tensor or numpy) -> resample back to the cropped grid (order 1, device) -> argmax (labels
    0 .. classes-1, ties to the lower class) -> paste into
    zeros(original size) at the crop box -> uint8 NIfTI with the input's header.  softmax_fname: the fork's
    `--save_softmax` (background probability as `<case>_0.nii.gz`, DCNN_multistage.py:340-343,359: 1 outside the crop);
    post3mm_fname: `remove_3mm_sparks` of the label map on the device (deepwmh/main/predict.py:19-26,158-163).
    for_which_classes / min_valid_object_sizes: a postprocessing.json (deepwmh_b200/postprocessing.py), applied on the
    device to the label file only, as upstream's predict_cases rewrites that file; the other outputs do not see it.
    region_class_order: a region-based model's order (softmax then holds its sigmoid probabilities); the labels are the
    region rule of SegmentationNetwork.region_labels on the resampled probabilities instead of the argmax.
    Returns the label map as written."""
    import torch

    from . import nifti, postprocessing
    hdr = properties["nifti_header"]
    with torch.cuda.device(network.device):
        sm = softmax if isinstance(softmax, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(softmax))
        sm = sm.to(device=network.device, dtype=torch.float32).contiguous()
        sm = resample_softmax_back_device(sm, properties["size_after_cropping"], properties["original_spacing"],
                                          properties["spacing_after_resampling"], force_separate_z, order)
        seg = network.argmax(sm.contiguous()) if region_class_order is None else network.region_labels(sm.contiguous(), region_class_order)
        full_shape = tuple(int(v) for v in properties["original_size_of_raw_data"])
        sl = tuple(slice(b[0], b[1]) for b in properties["crop_bbox"])
        full = torch.zeros(full_shape, dtype=torch.uint8, device=network.device)
        full[sl] = seg
        labels = full
        if for_which_classes:
            # [U:inference/predict.py::predict_cases -> load_remove_save]: sizes in mm^3 of the written image's spacing
            volume_per_voxel = float(np.prod(np.asarray(hdr["spacing"], dtype=np.float64)))
            labels = postprocessing.remove_all_but_the_largest_connected_component(network, full.clone(), for_which_classes,
                                                                                    volume_per_voxel, min_valid_object_sizes)
        nifti.write_nifti(out_fname, np.transpose(labels.cpu().numpy(), (2, 1, 0)), hdr, dtype=np.uint8)
        if post3mm_fname is not None:
            clean = network.remove_3mm_sparks(full.contiguous(), list(hdr["spacing"][::-1])).cpu().numpy()
            nifti.write_nifti(post3mm_fname, np.transpose(clean, (2, 1, 0)).astype(np.float32), hdr, dtype=np.float32)
        if softmax_fname is not None:
            bg = torch.ones(full_shape, dtype=torch.float32, device=network.device)
            bg[sl] = sm[0]
            nifti.write_nifti(softmax_fname, np.transpose(bg.cpu().numpy(), (2, 1, 0)), hdr, dtype=np.float32)
    return labels
