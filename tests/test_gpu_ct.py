"""CT models and nnU-Net's cascade on the B200 (DESIGN §13):
  * dwmh_ct_normalize "CT" bit for bit against the float32 restatement (odd sizes, n % 4 != 0, unaligned buffers, with and
    without the crop mask, planted lb / ub / +-1 ulp values); "CT2" within tolerance of the float64-statistics restatement,
    bit-identical repeats, its statistics, and the refusal of an empty mask;
  * dwmh_cascade_onehot bit for bit against resize_segmentation(order 1) + one-hot: up-, down- and equal-size grids, odd
    shapes, 2 .. 4 classes;
  * nnUNet_predict end to end on synthetic CT-like cases with random-init weights against the oracle pipeline: a one-modality
    three-class 3d_fullres CT model, two-stage plans through 3d_lowres, and 3d_cascade_fullres with -l and with the automatic
    low-resolution pass (identical labels), with a postprocessing.json in the cascade folder.
"""
import json
import os
import types

import numpy as np
import pytest
import torch

import ct_oracle as CO
import oracle as O
import postprocessing_oracle as PO
from deepwmh_b200 import nifti, preprocess
from deepwmh_b200 import nnunet_predict as NP
from test_host_ct import CT_PROPS, model_dir, two_stage_plans

pytestmark = pytest.mark.gpu

F32 = np.float32
PROB_TOL, AGREE_MIN = 2e-2, 0.999


def _planted(n, lb, ub, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(lb - 0.3 * (ub - lb), ub + 0.3 * (ub - lb), n).astype(F32)
    for v in (F32(lb), F32(ub)):
        for w in (v, np.nextafter(v, F32(np.inf)), np.nextafter(v, F32(-np.inf))):
            x[rng.random(n) < 0.03] = w
    seg = np.where(rng.random(n) < 0.2, -1, 0).astype(np.int8)
    return x, seg


def _device_ct(x, seg, scheme, c, offset=0):
    """dwmh_ct_normalize on a copy of x placed `offset` floats into a fresh buffer (offset 1: not 16-byte aligned)."""
    buf = torch.zeros(x.size + offset, dtype=torch.float32, device="cuda")
    v = buf[offset:]
    v.copy_(torch.from_numpy(x))
    s = None
    if seg is not None:
        sb = torch.zeros(seg.size + offset, dtype=torch.int8, device="cuda")
        s = sb[offset:]
        s.copy_(torch.from_numpy(seg))
    stats = preprocess.ct_normalize_device(v, s, scheme, c)
    return v.cpu().numpy(), stats


@pytest.mark.parametrize("n", [1, 3, 7, 1000, 4099, 37 * 41 * 29, 96 * 112 * 96])
def test_ct_is_the_float32_restatement_bit_for_bit(n):
    c = dict(CT_PROPS, mean=81.3, sd=117.9)
    lb, ub = c["percentile_00_5"], c["percentile_99_5"]
    x, seg = _planted(n, lb, ub, seed=n)
    for mask in (None, seg):
        want = CO.ct_normalize(x, lb, ub, c["mean"], c["sd"], mask)
        for offset in (0, 1):
            got, stats = _device_ct(x, mask, "CT", c, offset)
            assert stats is None
            bad = int((got != want).sum())
            assert bad == 0, (n, mask is not None, offset, bad)


@pytest.mark.parametrize("n", [5, 4099, 37 * 41 * 29, 182 * 218 * 182])
def test_ct2_matches_the_fp64_restatement_and_repeats_bit_for_bit(n):
    c = {"percentile_00_5": -1000.0, "percentile_99_5": 1500.0}
    lb, ub = c["percentile_00_5"], c["percentile_99_5"]
    x, seg = _planted(n, lb, ub, seed=7 + n)
    mn, sd, cnt = CO.ct2_stats(x, lb, ub)
    for mask in (None, seg):
        got, stats = _device_ct(x, mask, "CT2", c)
        again, stats2 = _device_ct(x, mask, "CT2", c)
        assert np.array_equal(got, again) and stats == stats2
        assert stats[2] == cnt and abs(stats[0] - mn) <= 1e-9 * abs(mn) + 1e-9 and abs(stats[1] - sd) <= 1e-9 * sd
        want = CO.ct2_normalize(x, lb, ub, mask)
        err = np.abs(got.astype(np.float64) - want).max()
        print("CT2 n=%d mask %s: max |x - x_ref| %.2e, mask count %d" % (n, mask is not None, err, cnt))
        assert err <= 1e-5 * max(1.0, np.abs(want).max())
        if mask is not None:
            assert (got[mask < 0] == 0).all()


def test_ct2_refuses_an_empty_mask_naming_case_and_modality(tmp_path):
    plans = two_stage_plans()
    plans["normalization_schemes"] = {0: "CT2"}
    plans["dataset_properties"]["intensityproperties"][0] = {"percentile_00_5": 100.0, "percentile_99_5": 200.0}
    vol = np.full((9, 10, 11), 50.0, np.float32)                   # every voxel below lb
    f = str(tmp_path / "liver_7_0000.nii.gz")
    nifti.write_nifti(f, vol, nifti.default_header(vol.shape))
    net = types.SimpleNamespace(device=torch.device("cuda", 0))
    with pytest.raises(ValueError, match="liver_7_0000.nii.gz, modality 0: no voxel lies strictly between the CT2 bounds"):
        preprocess.preprocess_test_case(net, plans, [f])


def _blobs(shape, num_classes, seed):
    """Smooth label regions (so the order-1 resize has edges to interpolate), labels 0 .. num_classes-1."""
    from scipy.ndimage import gaussian_filter
    rng = np.random.default_rng(seed)
    f = gaussian_filter(rng.normal(size=shape), 1.5)
    q = np.quantile(f, np.linspace(0, 1, num_classes + 1)[1:-1])
    return np.searchsorted(q, f).astype(np.uint8)


@pytest.mark.parametrize("src,dst", [((10, 12, 9), (17, 23, 15)), ((31, 26, 19), (14, 13, 11)), ((13, 14, 15), (13, 14, 15)),
                                     ((9, 20, 7), (18, 11, 7)), ((40, 33, 27), (41, 65, 27))])
@pytest.mark.parametrize("num_classes", [2, 3, 4])
def test_cascade_onehot_is_resize_segmentation_bit_for_bit(src, dst, num_classes):
    lab = _blobs(src, num_classes, seed=sum(src) + num_classes)
    want = CO.cascade_channels(lab, dst, num_classes)
    out = torch.full((num_classes - 1,) + dst, -7.0, dtype=torch.float32, device="cuda")
    preprocess.cascade_onehot_device(torch.from_numpy(lab).cuda(), out, num_classes)
    got = out.cpu().numpy()
    fr = [float(want[k].mean()) for k in range(num_classes - 1)]
    print("one-hot %s -> %s, C=%d: class fractions %s" % (src, dst, num_classes, fr))
    assert np.array_equal(got, want) and all(0 < v < 1 for v in fr)


# ---- nnUNet_predict end to end ---------------------------------------------------------------------------------------
SHAPE_ZYX, SPACING_ZYX = (40, 56, 48), (1.5, 1.0, 1.0)


def _ct_case(seed):
    """A CT-like volume in Hounsfield units: air everywhere (so the nonzero crop is the whole volume), a soft-tissue body,
    two brighter organs and a bone."""
    rng = np.random.default_rng(seed)
    z, y, x = np.meshgrid(*[np.linspace(-1, 1, s) for s in SHAPE_ZYX], indexing="ij")
    v = np.full(SHAPE_ZYX, -1000.0)
    v[(y / 0.8) ** 2 + (x / 0.9) ** 2 < 1] = 40.0
    v[((y - 0.2) / 0.35) ** 2 + ((x + 0.3) / 0.3) ** 2 + (z / 0.7) ** 2 < 1] = 150.0
    v[((y + 0.3) / 0.2) ** 2 + ((x - 0.35) / 0.25) ** 2 + ((z - 0.2) / 0.5) ** 2 < 1] = 260.0
    v[((y + 0.55) / 0.1) ** 2 + (x / 0.12) ** 2 < 1] = 900.0
    return (v + rng.normal(0, 25, SHAPE_ZYX)).astype(np.float32)


def _write_case(indir, case, vol):
    os.makedirs(indir, exist_ok=True)
    hdr = nifti.default_header(SHAPE_ZYX[::-1], spacing=SPACING_ZYX[::-1])
    nifti.write_nifti(os.path.join(indir, case + "_0000.nii.gz"), np.transpose(vol, (2, 1, 0)), hdr)
    return hdr


def _ct_plans():
    p = two_stage_plans(M=1, C=3)
    p["plans_per_stage"][1]["current_spacing"] = np.array([1.2, 1.0, 1.0])
    p["plans_per_stage"][0]["current_spacing"] = np.array([2.4, 2.0, 2.0])
    return p


def _read(path):
    return np.transpose(nifti.read_nifti(path)[0], (2, 1, 0))


def _compare(name, seg, bg, ref, p_ref):
    agree = float(np.mean(seg == ref))
    err = float(np.abs(bg - p_ref[0]).max())                        # the crop is the whole volume
    fr = [float((ref == c).mean()) for c in range(3)]
    print("%s: label agreement %.5f, max |p0 - p0_oracle| %.2e, oracle label fractions %s" % (name, agree, err, fr))
    assert agree >= AGREE_MIN and err <= PROB_TOL
    assert sum(f > 0.001 for f in fr) >= 2, fr                      # the agreement is not vacuous


def test_nnunet_predict_ct_fullres_lowres_and_cascade_end_to_end(tmp_path, monkeypatch):
    plans = _ct_plans()
    root = str(tmp_path / "model")
    net_full = O.build_benchmark_network(3, CO.stage_plans(plans, 1))
    net_low = O.build_benchmark_network(4, CO.stage_plans(plans, 0))
    casc_plans = dict(CO.stage_plans(plans, 1), num_modalities=3)  # 1 modality + 3 classes - 1
    net_casc = O.build_benchmark_network(5, casc_plans)
    model_dir(root, "3d_fullres", "nnUNetTrainerV2", plans, net_full.state_dict())
    model_dir(root, "3d_lowres", "nnUNetTrainerV2", plans, net_low.state_dict())
    cdir = model_dir(root, "3d_cascade_fullres", "nnUNetTrainerV2CascadeFullRes", plans, net_casc.state_dict())
    pp = {"for_which_classes": [1, 2]}
    with open(os.path.join(cdir, "postprocessing.json"), "w") as f:
        json.dump(pp, f)
    vol = _ct_case(0)
    indir = str(tmp_path / "in")
    hdr = _write_case(indir, "liver_1", vol)
    monkeypatch.setenv("RESULTS_FOLDER", root)
    base = ["-i", indir, "-t", "Task003_Liver", "-f", "all", "-chk", "model_best", "--save_softmax"]
    data = vol[None]

    # 3d_fullres: CT normalisation of a one-modality three-class model
    out = str(tmp_path / "full")
    assert NP.main(base + ["-o", out, "-m", "3d_fullres"]) == 0
    ref, p_ref = CO.predict_case(plans, net_full, data, SPACING_ZYX)
    _compare("3d_fullres CT", _read(os.path.join(out, "liver_1.nii.gz")), _read(os.path.join(out, "liver_1_0.nii.gz")), ref, p_ref)

    # 3d_lowres: the smallest stage's spacing and network
    out = str(tmp_path / "low")
    assert NP.main(base + ["-o", out, "-m", "3d_lowres"]) == 0
    low = _read(os.path.join(out, "liver_1.nii.gz"))
    ref, p_ref = CO.predict_case(plans, net_low, data, SPACING_ZYX, stage=0)
    _compare("3d_lowres CT", low, _read(os.path.join(out, "liver_1_0.nii.gz")), ref, p_ref)

    # 3d_cascade_fullres with -l, against the oracle fed the same previous-stage labels, then the postprocessing.json
    out_l = str(tmp_path / "casc_l")
    assert NP.main(base + ["-o", out_l, "-m", "3d_cascade_fullres", "-l", out]) == 0
    ref, p_ref = CO.predict_case(dict(plans), net_casc, data, SPACING_ZYX, seg_prev=low)
    ref_pp = PO.remove_all_but_the_largest_connected_component(ref, [1, 2], float(np.prod(hdr["spacing"])))
    seg_l = _read(os.path.join(out_l, "liver_1.nii.gz"))
    _compare("3d_cascade_fullres -l", seg_l, _read(os.path.join(out_l, "liver_1_0.nii.gz")), ref_pp, p_ref)
    assert json.load(open(os.path.join(out_l, "postprocessing.json"))) == pp

    # without -l: 3d_lowres first into <out>/3d_lowres_predictions, then the same labels
    out_a = str(tmp_path / "casc_auto")
    assert NP.main(base + ["-o", out_a, "-m", "3d_cascade_fullres"]) == 0
    assert np.array_equal(_read(os.path.join(out_a, "3d_lowres_predictions", "liver_1.nii.gz")), low)
    assert np.array_equal(_read(os.path.join(out_a, "liver_1.nii.gz")), seg_l)
