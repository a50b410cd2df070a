"""CPU side of CT models and the cascade (DESIGN §13): the float32 restatement's known answers, the plans' validation, every
refusal of dwmh_ct_normalize / dwmh_cascade_onehot through the C header, and nnUNet_predict's -m 3d_lowres /
3d_cascade_fullres argument handling -- all refused before any GPU work."""
import os
import pickle
import subprocess

import numpy as np
import pytest
import torch

import ct_oracle as CO
from conftest import small_plans
from deepwmh_b200 import _lib, nifti, preprocess
from deepwmh_b200 import nnunet_predict as NP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def test_ct_restatement_known_answers_at_the_bounds():
    lb, ub, mean, sd = -100.0, 200.0, 0.0, 0.5                  # x - 0 and x / 0.5 are exact
    up, down = (lambda v: np.nextafter(F32(v), F32(np.inf))), (lambda v: np.nextafter(F32(v), F32(-np.inf)))
    x = np.array([lb, down(lb), up(lb), ub, up(ub), down(ub), -1e6, 1e6, 0.0, np.nan], F32)
    y = CO.ct_normalize(x, lb, ub, mean, sd)
    assert y.dtype == np.float32
    assert (y[[0, 1, 6]] == F32(-200.0)).all() and (y[[3, 4, 7]] == F32(400.0)).all()   # clipped: exactly (bound - mean) / sd
    assert y[2] == (up(lb) - F32(mean)) / F32(sd) and y[2] > -200.0                      # one ulp inside stays inside
    assert y[5] == (down(ub) - F32(mean)) / F32(sd) and y[5] < 400.0
    assert y[8] == 0.0 and np.isnan(y[9])                                                # numpy.clip keeps NaN
    # float32 arithmetic with float32-rounded constants, not float64: 0.1 is not representable
    z = CO.ct_normalize(np.array([1.0], F32), -10.0, 10.0, 0.1, 0.3)
    assert z[0] == (F32(1.0) - F32(0.1)) / F32(0.3) and z[0] != F32((1.0 - 0.1) / 0.3)
    # use_mask_for_norm: zero where seg < 0, the rest untouched
    seg = np.array([0, -1, 0, -1, 0, 0, -1, 0, 0, 0], np.int8)
    ym = CO.ct_normalize(x, lb, ub, mean, sd, seg)
    assert (ym[seg < 0] == 0).all() and np.array_equal(ym[seg >= 0], y[seg >= 0], equal_nan=True)


def test_ct2_statistics_use_the_open_interval_of_the_unclipped_values():
    lb, ub = -100.0, 200.0
    up, down = (lambda v: np.nextafter(F32(v), F32(np.inf))), (lambda v: np.nextafter(F32(v), F32(-np.inf)))
    x = np.array([lb, ub, -500.0, 900.0, up(lb), down(ub), 10.0], F32)
    mn, sd, n = CO.ct2_stats(x, lb, ub)
    inside = np.array([up(lb), down(ub), 10.0], np.float64)
    assert n == 3 and mn == inside.mean() and sd == inside.std()
    y = CO.ct2_normalize(x, lb, ub)
    assert y[0] == y[2] == (F32(lb) - F32(mn)) / F32(sd) and y[1] == y[3] == (F32(ub) - F32(mn)) / F32(sd)
    assert abs(float(y[[4, 5, 6]].astype(np.float64).mean())) < 1e-6


def _ct_plans(schemes, props=None):
    p = small_plans()
    p["num_modalities"] = len(schemes)
    p["normalization_schemes"] = dict(enumerate(schemes))
    p["use_mask_for_norm"] = {m: False for m in range(len(schemes))}
    if props is not None:
        p["dataset_properties"] = {"intensityproperties": props}
    return p


CT_PROPS = {"mean": 80.0, "sd": 120.0, "percentile_00_5": -1000.0, "percentile_99_5": 1500.0}


def test_plans_validation_and_its_messages():
    got = preprocess.normalization_schemes(_ct_plans(["CT", "CT2", "noNorm", "nonCT"], {0: CT_PROPS, 1: {"percentile_00_5": -5, "percentile_99_5": 5}}))
    assert [s for s, _ in got] == ["CT", "CT2", "noNorm", "nonCT"]
    assert got[0][1] == CT_PROPS and got[1][1] == {"percentile_00_5": -5.0, "percentile_99_5": 5.0} and got[2][1] is None
    with pytest.raises(NotImplementedError, match=r"scheme 'CT' of modality 0 needs .*intensityproperties'\]\[0\]\['percentile_00_5'\]"):
        preprocess.normalization_schemes(_ct_plans(["CT"]))
    with pytest.raises(NotImplementedError, match=r"scheme 'CT' of modality 1 needs .*\['sd'\]"):
        preprocess.normalization_schemes(_ct_plans(["nonCT", "CT"], {1: {k: v for k, v in CT_PROPS.items() if k != "sd"}}))
    with pytest.raises(NotImplementedError, match=r"scheme 'CT2' of modality 0 needs .*\['percentile_99_5'\]"):
        preprocess.normalization_schemes(_ct_plans(["CT2"], {0: {"percentile_00_5": 1.0}}))
    with pytest.raises(NotImplementedError, match="scheme 'MRI' of modality 0: nnU-Net's nonCT, CT, CT2, noNorm"):
        preprocess.normalization_schemes(_ct_plans(["MRI"]))
    for bad in ({"percentile_00_5": 10.0, "percentile_99_5": -10.0}, {"percentile_00_5": float("nan")}, {"mean": float("inf")},
                {"percentile_99_5": 1e39}):
        with pytest.raises(ValueError, match="intensityproperties\\[0\\]"):
            preprocess.normalization_schemes(_ct_plans(["CT"], {0: dict(CT_PROPS, **bad)}))
    for sd in (0.0, -1.0, 1e-50):
        with pytest.raises(ValueError, match="'sd'.*divides"):
            preprocess.normalization_schemes(_ct_plans(["CT"], {0: dict(CT_PROPS, sd=sd)}))
    # the scheme check comes before any file is read: the input files need not exist
    with pytest.raises(NotImplementedError, match="'CT2' of modality 0"):
        preprocess.preprocess_test_case(None, _ct_plans(["CT2"]), ["missing_0000.nii.gz"])


def _run_c(tmp_path, body):
    _lib.load()
    src = tmp_path / "t.c"
    src.write_text('#include <math.h>\n#include <stdio.h>\n#include <stdint.h>\n#include "deepwmh_b200.h"\n'
                   "int main(void) {\n" + body + "\n  return 0;\n}\n")
    exe = str(tmp_path / "t")
    libdir = os.path.dirname(_lib.lib_path())
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src), "-L", libdir, "-ldeepwmh_b200",
                           "-Wl,-rpath," + libdir, "-lm"])
    return [l.split("|", 1) for l in subprocess.check_output([exe]).decode().splitlines()]


def test_ct_normalize_refusals_through_the_header(tmp_path):
    """Every refusal of dwmh_ct_normalize comes before any device work (the pointers are never dereferenced)."""
    res = _run_c(tmp_path, r'''
  float* v = (float*)(uintptr_t)0x1000; void* ws = (void*)(uintptr_t)0x2000; double st[3];
  #define T(...) { int rc = dwmh_ct_normalize(__VA_ARGS__); printf("%d|%s\n", rc, dwmh_last_error()); }
  T(0, 0, 0, 16, DWMH_NORM_CT, -1, 1, 0, 1, 0, 0, 0);
  T(0, v, 0, 0, DWMH_NORM_CT, -1, 1, 0, 1, 0, 0, 0);
  T(0, v, 0, -5, DWMH_NORM_CT2, -1, 1, 0, 1, 0, ws, 0);
  T(0, v, 0, 16, 0, -1, 1, 0, 1, 0, 0, 0);
  T(0, v, 0, 16, 3, -1, 1, 0, 1, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, 2, 1, 0, 1, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT2, 2, 1, 0, 1, 0, ws, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, NAN, 1, 0, 1, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT2, -1, INFINITY, 0, 1, 0, ws, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, -1, 1e39, 0, 1, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, -1, 1, NAN, 1, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, -1, 1, 0, INFINITY, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, -1, 1, 0, 0, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, -1, 1, 0, -2, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, -1, 1, 0, 1e-50, 0, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT, -1, 1, 0, 1, st, 0, 0);
  T(0, v, 0, 16, DWMH_NORM_CT2, -1, 1, 0, 1, st, 0, 0);
  T(0, (float*)(uintptr_t)0x1004, 0, 16, DWMH_NORM_CT2, -1, 1, 0, 1, st, ws, 0);
''')
    assert all(rc != "0" for rc, _ in res) and len(res) == 18
    msgs = [m for _, m in res]
    assert "null vol" in msgs[0]
    assert "n=0 (must be > 0)" in msgs[1] and "n=-5" in msgs[2]
    assert "unknown scheme 0" in msgs[3] and "unknown scheme 3" in msgs[4]
    assert "lb=2 > ub=1" in msgs[5] and "lb=2 > ub=1" in msgs[6]
    assert all("must be finite in fp32" in m for m in msgs[7:12])
    assert all("sd=" in m and "must be > 0" in m for m in msgs[12:15])
    assert "stats_out is for CT2 only" in msgs[15]
    assert "CT2 needs a workspace" in msgs[16] and "aligned" in msgs[17]


def test_cascade_onehot_refusals_through_the_header(tmp_path):
    res = _run_c(tmp_path, r'''
  const uint8_t* l = (const uint8_t*)(uintptr_t)0x1000; float* d = (float*)(uintptr_t)0x2000;
  int32_t s[3] = {4, 5, 6}, z0[3] = {0, 5, 6}, z2[3] = {4, 5, -1};
  #define T(...) { int rc = dwmh_cascade_onehot(__VA_ARGS__); printf("%d|%s\n", rc, dwmh_last_error()); }
  T(0, 0, s, d, s, 3, 0);
  T(0, l, s, 0, s, 3, 0);
  T(0, l, 0, d, s, 3, 0);
  T(0, l, s, d, 0, 3, 0);
  T(0, l, s, d, s, 1, 0);
  T(0, l, s, d, s, 9, 0);
  T(0, l, z0, d, s, 3, 0);
  T(0, l, s, d, z2, 3, 0);
''')
    assert all(rc != "0" for rc, _ in res) and len(res) == 8
    msgs = [m for _, m in res]
    assert all("null argument" in m for m in msgs[:4])
    assert "num_classes=1 unsupported (2 <= num_classes <= 8)" in msgs[4] and "num_classes=9 unsupported" in msgs[5]
    assert "empty extent on axis 0" in msgs[6] and "empty extent on axis 2" in msgs[7]


# ---- nnUNet_predict -m 3d_lowres / 3d_cascade_fullres -----------------------------------------------------------------
def two_stage_plans(M=1, C=3):
    p = small_plans()
    p["num_modalities"], p["num_classes"] = M, C - 1
    p["normalization_schemes"] = {m: "CT" for m in range(M)}
    p["use_mask_for_norm"] = {m: False for m in range(M)}
    p["dataset_properties"] = {"intensityproperties": {m: dict(CT_PROPS) for m in range(M)}}
    low = dict(p["plans_per_stage"][0], current_spacing=np.array([2.0, 2.0, 2.0]))
    p["plans_per_stage"] = {0: low, 1: p["plans_per_stage"][0]}
    return p


def model_dir(root, model, trainer, plans, state_dict=None, task="Task003_Liver"):
    tdir = os.path.join(root, "nnUNet", model, task, "%s__nnUNetPlansv2.1" % trainer)
    os.makedirs(os.path.join(tdir, "all"), exist_ok=True)
    pickle.dump(plans, open(os.path.join(tdir, "plans.pkl"), "wb"))
    if state_dict is None:
        open(os.path.join(tdir, "all", "model_best.model"), "wb").close()
    else:
        torch.save({"epoch": 1, "state_dict": state_dict}, os.path.join(tdir, "all", "model_best.model"))
    return tdir


def _inputs(indir, M=1, shape=(12, 10, 8), cases=("c1",)):
    os.makedirs(indir, exist_ok=True)
    hdr = nifti.default_header(shape)
    for c in cases:
        for m in range(M):
            nifti.write_nifti(os.path.join(indir, "%s_%04d.nii.gz" % (c, m)), np.ones(shape, np.float32), hdr)
    return hdr


def test_nnunet_predict_cascade_refusals_before_any_gpu_work(tmp_path, monkeypatch):
    root = str(tmp_path / "m")
    plans = two_stage_plans()
    one_stage = small_plans()
    model_dir(root, "3d_lowres", "nnUNetTrainerV2", plans)
    model_dir(root, "3d_cascade_fullres", "nnUNetTrainerV2CascadeFullRes", plans)
    model_dir(root, "3d_lowres", "nnUNetTrainerV2", one_stage, task="Task004_Single")
    big = two_stage_plans(M=2, C=4)                              # 2 + 4 - 1 = 5 input channels
    model_dir(root, "3d_cascade_fullres", "nnUNetTrainerV2CascadeFullRes", big, task="Task005_Big")
    indir = str(tmp_path / "in")
    hdr = _inputs(indir)
    lowdir = tmp_path / "low"; lowdir.mkdir()
    monkeypatch.setenv("RESULTS_FOLDER", root)
    out = str(tmp_path / "o")
    base = ["-i", indir, "-o", out, "-f", "all", "-chk", "model_best"]
    with pytest.raises(RuntimeError, match="one plans stage, so it has no 3d_lowres stage"):
        NP.main(base + ["-t", "Task004_Single", "-m", "3d_lowres"])
    with pytest.raises(RuntimeError, match="previous stage's segmentation .*c1.nii.gz does not exist"):
        NP.main(base + ["-t", "Task003_Liver", "-m", "3d_cascade_fullres", "-l", str(lowdir)])
    lab = np.zeros((12, 10, 8), np.float32)
    lab[3, 3, 3] = 3.0                                           # the model has labels 0 .. 2
    nifti.write_nifti(str(lowdir / "c1.nii.gz"), lab, hdr, dtype=np.uint8)
    with pytest.raises(ValueError, match=r"holds values 3 outside the labels 0 .. 2"):
        NP.main(base + ["-t", "Task003_Liver", "-m", "3d_cascade_fullres", "-l", str(lowdir)])
    nifti.write_nifti(str(lowdir / "c1.nii.gz"), lab[:11], nifti.default_header((11, 10, 8)), dtype=np.uint8)
    with pytest.raises(ValueError, match=r"has shape \(11, 10, 8\), the case's images \(12, 10, 8\)"):
        NP.main(base + ["-t", "Task003_Liver", "-m", "3d_cascade_fullres", "-l", str(lowdir)])
    with pytest.raises(NotImplementedError, match="= 5 input channels; at most DWMH_MAX_IN_CHANNELS = 4"):
        NP.main(base + ["-t", "Task005_Big", "-m", "3d_cascade_fullres", "-l", str(lowdir)])
    with pytest.raises(ValueError, match="needs --part_id 0 --num_parts 1"):
        NP.main(base + ["-t", "Task003_Liver", "-m", "3d_cascade_fullres", "--num_parts", "2"])
    with pytest.raises(NotImplementedError, match="serves -ctr nnUNetTrainerV2CascadeFullRes only"):
        NP.main(base + ["-t", "Task003_Liver", "-m", "3d_cascade_fullres", "-ctr", "nnUNetTrainerCascadeFullRes"])
    with pytest.raises(NotImplementedError, match="-l .* 3d_cascade_fullres only"):
        NP.main(base + ["-t", "Task003_Liver", "-m", "3d_lowres", "-l", str(lowdir)])
    with pytest.raises(NotImplementedError, match="serves -tr nnUNetTrainerV2 .* -m 3d_fullres \\| 3d_lowres \\| 3d_cascade_fullres"):
        NP.main(base + ["-t", "Task003_Liver", "-m", "2d"])
    # the automatic low-resolution pass needs its own model folder, named by -tr
    with pytest.raises(RuntimeError, match="3d_lowres.*nnUNetTrainerV2BraTSRegions__nnUNetPlansv2.1.*plans.pkl"):
        NP.main(base + ["-t", "Task003_Liver", "-m", "3d_cascade_fullres", "-tr", "nnUNetTrainerV2BraTSRegions"])
    assert not os.path.exists(out)


def test_stages_of_each_configuration(tmp_path):
    plans = two_stage_plans()
    root = str(tmp_path)
    for model, want in (("3d_lowres", 0), ("3d_cascade_fullres", 1), ("3d_fullres", 1)):
        tdir = model_dir(root, model, "T", plans)
        _, _, stage = NP._load_model(tdir, os.path.join(tdir, "plans.pkl"), os.path.join(tdir, "all", "%s.model"), "model_best", model)
        assert stage == want, model
    tdir = model_dir(root, "3d_fullres", "T", small_plans(), task="Task009_One")
    assert NP._load_model(tdir, os.path.join(tdir, "plans.pkl"), os.path.join(tdir, "all", "%s.model"), "model_best", "3d_fullres")[2] == 0
