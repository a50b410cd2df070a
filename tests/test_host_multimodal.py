"""CPU side of multi-modality / multi-class models: case discovery, the oracle pipeline's union mask and per-modality
z-score, dwmh_create's model bounds through the C header, and DeepWMH_predict's refusal of multi-modality models."""
import os
import pickle
import subprocess

import numpy as np
import pytest

import oracle as O
import oracle.resample_oracle as R
from conftest import small_plans
from deepwmh_b200 import _lib, cli, preprocess
from deepwmh_b200 import nnunet_predict as NP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _touch(p):
    open(p, "wb").close()


def test_case_files_lists_modalities_in_order_and_names_the_missing_one(tmp_path):
    for f in ("a_0000.nii.gz", "a_0001.nii.gz", "a_0002.nii.gz", "b_0000.nii.gz", "b_0002.nii.gz"):
        _touch(tmp_path / f)
    assert NP._cases_in(str(tmp_path)) == ["a", "b"]
    assert [os.path.basename(f) for f in NP.case_files(str(tmp_path), "a", 3)] == ["a_0000.nii.gz", "a_0001.nii.gz", "a_0002.nii.gz"]
    assert [os.path.basename(f) for f in NP.case_files(str(tmp_path), "b", 1)] == ["b_0000.nii.gz"]
    with pytest.raises(RuntimeError, match="case b lacks modality file.*b_0001.nii.gz"):
        NP.case_files(str(tmp_path), "b", 3)


def test_nnunet_predict_rejects_a_case_without_all_modalities_before_any_gpu_work(tmp_path, monkeypatch):
    plans = small_plans()
    plans["num_modalities"] = 2
    tdir = tmp_path / "m" / "nnUNet" / "3d_fullres" / "Task005_WMH" / "nnUNetTrainerV2__nnUNetPlansv2.1"
    (tdir / "all").mkdir(parents=True)
    pickle.dump(plans, open(tdir / "plans.pkl", "wb"))
    _touch(tdir / "all" / "model_best.model")
    indir = tmp_path / "in"; indir.mkdir()
    _touch(indir / "c1_0000.nii.gz"); _touch(indir / "c1_0001.nii.gz"); _touch(indir / "c2_0000.nii.gz")
    monkeypatch.setenv("RESULTS_FOLDER", str(tmp_path / "m"))
    with pytest.raises(RuntimeError, match="c2 lacks modality file.*c2_0001"):
        NP.main(["-i", str(indir), "-o", str(tmp_path / "o"), "-t", "Task005_WMH", "-f", "all", "-chk", "model_best"])
    assert not (tmp_path / "o").exists()


def test_read_modalities_requires_one_geometry(tmp_path):
    from deepwmh_b200 import nifti
    a = np.random.default_rng(0).random((6, 5, 4)).astype(np.float32)
    nifti.write_nifti(str(tmp_path / "x_0000.nii.gz"), a, nifti.default_header(a.shape, (1.0, 1.0, 2.0)))
    nifti.write_nifti(str(tmp_path / "x_0001.nii.gz"), 2 * a, nifti.default_header(a.shape, (1.0, 1.0, 2.0)))
    nifti.write_nifti(str(tmp_path / "x_0002.nii.gz"), a, nifti.default_header(a.shape, (1.0, 1.0, 3.0)))
    nifti.write_nifti(str(tmp_path / "x_0003.nii.gz"), a[:5], nifti.default_header(a[:5].shape, (1.0, 1.0, 2.0)))
    data, hdr = preprocess.read_modalities([str(tmp_path / "x_0000.nii.gz"), str(tmp_path / "x_0001.nii.gz")])
    assert data.shape == (2, 4, 5, 6) and np.array_equal(data[1], 2 * np.transpose(a, (2, 1, 0)))
    with pytest.raises(ValueError, match="geometry"):
        preprocess.read_modalities([str(tmp_path / "x_0000.nii.gz"), str(tmp_path / "x_0002.nii.gz")])
    with pytest.raises(ValueError, match="shape"):
        preprocess.read_modalities([str(tmp_path / "x_0000.nii.gz"), str(tmp_path / "x_0003.nii.gz")])


def test_union_nonzero_mask_and_per_modality_zscore():
    rng = np.random.default_rng(1)
    d = np.zeros((2, 12, 14, 10), np.float32)
    d[0, 2:8, 3:9, 2:7] = rng.normal(100, 20, (6, 6, 5))
    d[1, 5:11, 4:12, 3:9] = rng.normal(5, 1, (6, 8, 6))
    d[0, 4, 5, 4] = 0.0                                          # a hole inside the union: filled
    cropped, seg, bbox = preprocess.crop_to_nonzero(d)
    assert bbox == [[2, 11], [3, 12], [2, 9]]
    union = (d[0] != 0) | (d[1] != 0)
    inside = seg[0] == 0
    assert inside.sum() >= union[2:11, 3:12, 2:9].sum() and inside[2, 2, 2]
    out, s = R.resample_and_normalize(cropped, seg, [1.0, 1.0, 1.0], [1.0, 1.0, 1.0], True)
    for c in range(2):
        v = cropped[c][inside]
        ref = (cropped[c] - v.mean()) / (v.std() + 1e-8)
        assert np.allclose(out[c][inside], ref[inside], atol=1e-4)
        assert abs(out[c][inside].mean()) < 1e-4 and abs(out[c][inside].std() - 1.0) < 1e-3
        assert (out[c][~inside] == 0).all()


def test_preprocess_rejects_ct_normalisation_and_a_wrong_file_count():
    plans = small_plans()
    plans["num_modalities"] = 2
    plans["normalization_schemes"] = {0: "nonCT", 1: "CT"}
    with pytest.raises(ValueError, match="2 modalities; got 1"):
        preprocess.preprocess_test_case(None, plans, ["a_0000.nii.gz"])
    with pytest.raises(NotImplementedError, match="CT"):
        preprocess.preprocess_test_case(None, plans, ["a_0000.nii.gz", "a_0001.nii.gz"])


def test_create_bounds_through_the_header(tmp_path):
    """dwmh_create refuses in_channels outside 1..4, num_classes outside 2..8 (before any device work), naming the bound."""
    _lib.load()
    src = tmp_path / "b.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "deepwmh_b200.h"
int main(void) {
  const int cases[][2] = {{0, 2}, {5, 2}, {1, 1}, {1, 9}, {2, 0}};
  printf("%d %d\n", DWMH_MAX_IN_CHANNELS, DWMH_MAX_CLASSES);
  for (int i = 0; i < 5; ++i) {
    dwmh_net_desc d; memset(&d, 0, sizeof d);
    d.in_channels = cases[i][0]; d.num_classes = cases[i][1]; d.base_num_features = 32; d.num_pool = 1;
    d.struct_size = (int32_t)sizeof d;
    dwmh_ctx* c = 0;
    int rc = dwmh_create(&c, 0, &d);
    printf("%d|%s\n", rc, dwmh_last_error());
  }
  return 0;
}
''')
    exe = str(tmp_path / "b")
    libdir = os.path.dirname(_lib.lib_path())
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src), "-L", libdir, "-ldeepwmh_b200",
                           "-Wl,-rpath," + libdir])
    lines = subprocess.check_output([exe]).decode().splitlines()
    assert lines[0] == "%d %d" % (_lib.DWMH_MAX_IN_CHANNELS, _lib.DWMH_MAX_CLASSES) == "4 8"
    res = [l.split("|", 1) for l in lines[1:]]
    assert all(rc != "0" for rc, _ in res)
    assert "in_channels=0 unsupported (1 <= in_channels <= 4" in res[0][1]
    assert "in_channels=5 unsupported (1 <= in_channels <= 4" in res[1][1]
    assert "num_classes=1 unsupported (2 <= num_classes <= 8" in res[2][1]
    assert "num_classes=9 unsupported (2 <= num_classes <= 8" in res[3][1]
    assert "num_classes=0 unsupported" in res[4][1]


def test_deepwmh_predict_refuses_a_multi_modality_model(tmp_path):
    plans = small_plans()
    plans["num_modalities"] = 2
    tdir = tmp_path / "m" / "nnUNet" / "3d_fullres" / "Task005_WMH" / "nnUNetTrainerV2__nnUNetPlansv2.1"
    (tdir / "all").mkdir(parents=True)
    pickle.dump(plans, open(tdir / "plans.pkl", "wb"))
    _touch(tdir / "all" / "model_best.model")
    img = tmp_path / "flair.nii.gz"; _touch(img)
    with pytest.raises(RuntimeError, match="takes 2 input modalities.*nnUNet_predict"):
        cli.main(["-i", str(img), "-n", "c1", "-m", str(tmp_path / "m"), "-o", str(tmp_path / "o"), "--skip-bfc"])
    assert not (tmp_path / "o").exists()


def test_benchmark_plans_defaults_are_deepwmh_and_extend_to_m_c():
    from deepwmh_b200 import plans as P
    assert P.benchmark_plans()["num_modalities"] == 1 and P.benchmark_plans()["num_classes"] == 1
    p = P.benchmark_plans(num_modalities=2, num_classes=3)
    assert p["num_modalities"] == 2 and p["num_classes"] == 2 and set(p["use_mask_for_norm"]) == {0, 1}
    assert O.build_network(p).conv_blocks_context[0].blocks[0].conv.weight.shape[1] == 2
