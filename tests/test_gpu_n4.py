"""N4 bias-field correction on the device (dwmh_n4, deepwmh_b200.n4) against the fp64 restatement of oracle/n4_oracle.py
with DeepWMH's schedule (-s 2, 50x50x50x50), its determinism, its tensor / in-place forms, and DeepWMH_predict --device-bfc
end to end."""
import ctypes as C
import os
import pickle

import numpy as np
import pytest
import torch

import oracle as O
from conftest import small_plans
from deepwmh_b200 import _lib, cli, nifti
from deepwmh_b200.n4 import n4_bias_field_correction
from oracle import n4_oracle as N

SCHEDULE = (50, 50, 50, 50)
TOL = 1e-4


def _compare(img, out, field, ref_out, ref_field):
    v = img > 0
    d_field = float(np.abs(field.astype(np.float64) - ref_field).max())
    d_out = float((np.abs(out.astype(np.float64) - ref_out)[v] / np.abs(ref_out[v])).max())
    return d_field, d_out


def test_workspace_rejects_bad_extents():
    lib = _lib.load()
    b = C.c_int64()
    _lib.check(lib.dwmh_n4_workspace(182, 218, 182, 2, 4, C.byref(b)))
    assert b.value > 2 * 91 * 109 * 91 * 4
    for args in ((3, 64, 64, 2, 4), (64, 64, 64, 0, 4), (64, 64, 64, 2, 0), (64, 64, 64, 2, 9), (0, 8, 8, 1, 1)):
        with pytest.raises(_lib.DwmhError):
            _lib.check(lib.dwmh_n4_workspace(*args, C.byref(b)))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,seed", [((96, 112, 96), 0), ((161, 191, 41), 1)])
def test_device_matches_oracle(shape, seed):
    img, _, _ = N.phantom(shape, seed=seed)
    ref_out, ref_field = N.n4(img, 2, SCHEDULE, return_log_field=True)
    out, field = n4_bias_field_correction(img, 2, SCHEDULE, device=0, return_log_field=True)
    assert out.dtype == np.float32 and field.dtype == np.float32 and out.shape == img.shape
    d_field, d_out = _compare(img, out, field, ref_out, ref_field)
    print("n4 %s: log field max |d| %.3e, corrected max rel |d| %.3e" % (shape, d_field, d_out))
    assert d_field <= TOL and d_out <= TOL
    assert np.array_equal(out[img == 0], img[img == 0])


@pytest.mark.gpu
def test_two_calls_and_in_place_are_bit_identical():
    img, _, _ = N.phantom((80, 72, 64), seed=4)
    a, fa = n4_bias_field_correction(img, 2, (20, 20, 20), return_log_field=True)
    b, fb = n4_bias_field_correction(img, 2, (20, 20, 20), return_log_field=True)
    assert np.array_equal(a, b) and np.array_equal(fa, fb)
    lib = _lib.load()
    t = torch.from_numpy(img).cuda()
    nb = C.c_int64()
    _lib.check(lib.dwmh_n4_workspace(80, 72, 64, 2, 3, C.byref(nb)))
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    it = (C.c_int32 * 3)(20, 20, 20)
    _lib.check(lib.dwmh_n4(0, C.c_void_p(t.data_ptr()), 80, 72, 64, 2, 3, it, C.c_void_p(t.data_ptr()), None,
                           C.c_void_p(ws.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert np.array_equal(t.cpu().numpy(), a)


@pytest.mark.gpu
def test_cuda_tensor_stays_on_the_device():
    img, _, _ = N.phantom((64, 70, 50), seed=5)
    t = torch.from_numpy(img).cuda()
    out, field = n4_bias_field_correction(t, 2, (10, 10, 10), return_log_field=True)
    assert isinstance(out, torch.Tensor) and out.is_cuda and field.is_cuda and out.dtype == torch.float32
    ref, ref_f = n4_bias_field_correction(img, 2, (10, 10, 10), return_log_field=True)
    assert np.array_equal(out.cpu().numpy(), ref) and np.array_equal(field.cpu().numpy(), ref_f)
    assert torch.equal(t, torch.from_numpy(img).cuda())                      # the input is not modified


def _model_dir(root, plans, net):
    tdir = os.path.join(root, "nnUNet", "3d_fullres", "Task002_FinalModel", "nnUNetTrainerV2__nnUNetPlansv2.1")
    os.makedirs(os.path.join(tdir, "all"))
    pickle.dump(plans, open(os.path.join(tdir, "plans.pkl"), "wb"))
    torch.save({"epoch": 1, "state_dict": net.state_dict()}, os.path.join(tdir, "all", "model_best.model"))


@pytest.mark.gpu
def test_cli_device_bfc_end_to_end(tmp_path, monkeypatch):
    """DeepWMH_predict --device-bfc with no N4BiasFieldCorrection on PATH: the pre-processed image is the oracle's N4 of the
    input (-s 2, 50x50x50x50) with the input's header, and the segmentation files exist."""
    monkeypatch.setenv("PATH", str(tmp_path / "empty_bin"))
    plans = small_plans()
    plans["use_mask_for_norm"] = {0: True}
    net = O.build_benchmark_network(0, plans)
    root = str(tmp_path / "model")
    _model_dir(root, plans, net)
    vol_zyx = np.zeros((44, 52, 48), np.float32)
    vol_zyx[4:42, 6:50, 5:45] = O.synthetic_flair((38, 44, 40), seed=11)[0]
    vol_zyx[4:42, 6:50, 5:45][vol_zyx[4:42, 6:50, 5:45] == 0] = 3.0
    vol = np.ascontiguousarray(np.transpose(vol_zyx, (2, 1, 0)))
    img = str(tmp_path / "case1.nii.gz")
    nifti.write_nifti(img, vol, nifti.default_header(vol.shape, spacing=(0.9, 1.1, 3.0)))
    out = str(tmp_path / "out")
    assert cli.main(["-i", img, "-n", "case1", "-m", root, "-o", out, "--device-bfc", "-g", "0"]) == 0
    pre, hdr = nifti.read_nifti(os.path.join(out, "001_Preprocessed_Images", "case1_0000.nii.gz"))
    assert pre.dtype == np.float32 and pre.shape == vol.shape
    assert np.allclose(hdr["spacing"], (0.9, 1.1, 3.0))
    ref = N.n4(vol, 2, SCHEDULE)
    v = vol > 0
    assert float((np.abs(pre.astype(np.float64) - ref)[v] / np.abs(ref[v])).max()) <= TOL
    assert np.array_equal(pre[~v], vol[~v])
    for sub in ("001_raw", "002_postproc_3mm"):
        assert os.path.isfile(os.path.join(out, "002_Segmentations", sub, "case1.nii.gz"))
