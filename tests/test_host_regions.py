"""CPU side of region-based models (nnUNetTrainerV2BraTSRegions, DESIGN §12): the region rule of the restated reference
(tests/regions_oracle.py) on known answers, the trainer constants, dwmh_create's head_nonlin bound and dwmh_region_labels'
refusals through the C ABI, and nnUNet_predict's refusals before any GPU work."""
import ctypes as C
import os
import pickle
import subprocess

import numpy as np
import pytest
import torch

import regions_oracle as RO
from conftest import small_plans
from deepwmh_b200 import _lib
from deepwmh_b200 import nnunet_predict as NP
from deepwmh_b200.predictor import SegmentationNetwork, nnUNetTrainerV2, nnUNetTrainerV2BraTSRegions

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _upstream_loop(probs, order):
    """The rule voxel by voxel, as a literal reading of upstream's `seg[class_probabilities[i] > 0.5] = c` loop."""
    out = np.zeros(probs.shape[1:], np.float32)
    for idx in np.ndindex(*probs.shape[1:]):
        for i, c in enumerate(order):
            if probs[(i,) + idx] > 0.5:
                out[idx] = c
    return out


def test_region_rule_known_answers():
    half = np.float32(0.5)
    up, down = np.nextafter(half, np.float32(1)), np.nextafter(half, np.float32(0))
    # voxels: nested whole > core > enhancing; whole only; core without whole (a later region overwrites); exactly 0.5;
    # 0.5 + 1 ulp; 0.5 - 1 ulp; NaN in the last region; nothing
    p = np.array([
        [0.9, 0.9, 0.1, half, up, 0.9, 0.9, 0.0],
        [0.8, 0.2, 0.7, half, up, down, 0.9, 0.0],
        [0.7, 0.1, 0.2, half, up, 0.1, np.nan, 0.0],
    ], np.float32)
    want = np.array([3, 1, 2, 0, 3, 1, 2, 0], np.float32)
    got = RO.region_labels(p, RO.BRATS_REGIONS_CLASS_ORDER)
    assert got.dtype == np.float32 and np.array_equal(got, want)
    assert np.array_equal(_upstream_loop(p, (1, 2, 3)), want)
    # another order: the last listed region wins where several are inside
    assert np.array_equal(RO.region_labels(p, (3, 2, 1)), _upstream_loop(p, (3, 2, 1)))
    assert RO.region_labels(p, (3, 2, 1))[0] == 1
    rng = np.random.default_rng(0)
    q = rng.random((3, 5, 6, 7)).astype(np.float32)
    q[rng.random(q.shape) < 0.1] = half
    assert np.array_equal(RO.region_labels(q, (1, 2, 3)), _upstream_loop(q, (1, 2, 3)))


def test_region_oracle_predict_is_the_rule_on_its_probabilities():
    plans = small_plans()
    plans["num_modalities"] = 4
    net = RO.build_region_network(plans, 1)
    assert net.num_classes == 3 and net.seg_outputs[-1].weight.shape == (3, 32, 1, 1, 1)
    x = np.random.default_rng(2).normal(size=(4, 40, 36, 34)).astype(np.float32)
    seg, p = RO.predict_3D(net, x, False, (), 0.5, (32, 32, 32), RO.BRATS_REGIONS_CLASS_ORDER)
    assert seg.dtype == np.float32 and p.shape == (3, 40, 36, 34)
    assert p.min() > 0 and p.max() < 1 and not np.allclose(p.sum(0), 1.0)          # a sigmoid per output, no softmax
    assert np.array_equal(seg, RO.region_labels(p, (1, 2, 3)))
    seg_n, p_n = RO.predict_3D(net, x, False, (), 0.5, (32, 32, 32), None)
    assert np.array_equal(p_n, p) and np.array_equal(seg_n, p.argmax(0))


def test_brats_region_trainer_constants():
    T = nnUNetTrainerV2BraTSRegions
    assert T.regions == {"whole tumor": (1, 2, 3), "tumor core": (2, 3), "enhancing tumor": (3,)}
    assert T.regions_class_order == (1, 2, 3) and T.inference_nonlin == "sigmoid"
    assert nnUNetTrainerV2.regions_class_order is None and nnUNetTrainerV2.inference_nonlin == "softmax"
    assert RO.BRATS_REGIONS == T.regions and RO.BRATS_REGIONS_CLASS_ORDER == T.regions_class_order
    import deepwmh_b200
    assert deepwmh_b200.nnUNetTrainerV2BraTSRegions is T and "nnUNetTrainerV2BraTSRegions" in deepwmh_b200.__all__
    plans = small_plans()
    plans["num_modalities"], plans["num_classes"] = 4, 3                          # labels 1..3, three region outputs
    tr = T.__new__(T)
    tr.process_plans(plans)
    assert tr.num_classes == 3 and tr.num_input_channels == 4
    base = nnUNetTrainerV2.__new__(nnUNetTrainerV2)
    base.process_plans(plans)
    assert base.num_classes == 4


def test_segmentation_network_refuses_an_unknown_nonlinearity():
    with pytest.raises(ValueError, match="inference_nonlin must be one of"):
        SegmentationNetwork(small_plans(), inference_nonlin="softmax2")


def test_create_refuses_head_nonlin_outside_0_1_through_the_header(tmp_path):
    _lib.load()
    src = tmp_path / "h.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "deepwmh_b200.h"
int main(void) {
  const int v[] = {2, -1, 0, 1};
  for (int i = 0; i < 4; ++i) {
    dwmh_net_desc d; memset(&d, 0, sizeof d);
    d.in_channels = 4; d.num_classes = 3; d.base_num_features = 32; d.num_pool = 1; d.head_nonlin = v[i];
    d.struct_size = (int32_t)sizeof d;
    dwmh_ctx* c = 0;
    int rc = dwmh_create(&c, 0, &d);
    printf("%d|%s\n", rc, rc ? dwmh_last_error() : "");
    if (!rc) dwmh_destroy(c);
  }
  return 0;
}
''')
    exe = str(tmp_path / "h")
    libdir = os.path.dirname(_lib.lib_path())
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src), "-L", libdir, "-ldeepwmh_b200",
                           "-Wl,-rpath," + libdir])
    res = [l.split("|", 1) for l in subprocess.check_output([exe]).decode().splitlines()]
    assert res[0][0] != "0" and "head_nonlin=2 unsupported (0 = softmax over classes, 1 = sigmoid per output)" in res[0][1]
    assert res[1][0] != "0" and "head_nonlin=-1 unsupported" in res[1][1]
    assert all("head_nonlin" not in msg for _, msg in res[2:])                    # 0 and 1 pass the model bounds


def test_region_labels_refusals_need_no_device():
    """Every refusal happens before the context is used or any device work is enqueued: stand-in pointers suffice."""
    lib = _lib.load()
    buf = (C.c_uint8 * 64)()
    ctx, probs, seg = C.c_void_p(C.addressof(buf)), C.c_void_p(C.addressof(buf) + 16), C.c_void_p(C.addressof(buf) + 32)
    order = (C.c_int32 * 9)(1, 2, 3, 4, 5, 6, 7, 8, 9)

    def err(*args):
        assert lib.dwmh_region_labels(*args) != 0
        return lib.dwmh_last_error().decode()

    assert "null argument" in err(None, probs, 3, order, seg, 10, None)
    assert "null argument" in err(ctx, None, 3, order, seg, 10, None)
    assert "null argument" in err(ctx, probs, 3, None, seg, 10, None)
    assert "null argument" in err(ctx, probs, 3, order, None, 10, None)
    assert "num_regions=0 outside 1..8" in err(ctx, probs, 0, order, seg, 10, None)
    assert "num_regions=9 outside 1..8" in err(ctx, probs, 9, order, seg, 10, None)
    assert "region 1 has label 256" in err(ctx, probs, 3, (C.c_int32 * 3)(1, 256, 3), seg, 10, None)
    assert "region 0 has label -1" in err(ctx, probs, 3, (C.c_int32 * 3)(-1, 2, 3), seg, 10, None)
    assert "nvox=0" in err(ctx, probs, 3, order, seg, 0, None)
    assert "nvox=-5" in err(ctx, probs, 3, order, seg, -5, None)


def _model_dir(root, plans, trainer, state_dict=None):
    tdir = os.path.join(root, "nnUNet", "3d_fullres", "Task001_BrainTumour", "%s__nnUNetPlansv2.1" % trainer)
    os.makedirs(os.path.join(tdir, "all"), exist_ok=True)
    pickle.dump(plans, open(os.path.join(tdir, "plans.pkl"), "wb"))
    if state_dict is None:
        open(os.path.join(tdir, "all", "model_best.model"), "wb").close()
    else:
        torch.save({"epoch": 1, "state_dict": state_dict}, os.path.join(tdir, "all", "model_best.model"))
    return tdir


def test_nnunet_predict_refusals_before_any_gpu_work(tmp_path, monkeypatch):
    plans = small_plans()
    plans["num_modalities"], plans["num_classes"] = 4, 3
    root = str(tmp_path / "m")
    _model_dir(root, plans, "nnUNetTrainerV2BraTSRegions")
    indir = tmp_path / "in"; indir.mkdir()
    for m in range(4):
        open(indir / ("c1_%04d.nii.gz" % m), "wb").close()
    monkeypatch.setenv("RESULTS_FOLDER", root)
    base = ["-i", str(indir), "-o", str(tmp_path / "o"), "-t", "Task001_BrainTumour", "-f", "all", "-chk", "model_best"]
    for name in ("nnUNetTrainerV2BraTSRegions_BN", "nnUNetTrainerV2BraTSRegions_DA4_BN_BD", "nnUNetTrainerV2BraTSRegions_DA3_BN"):
        with pytest.raises(NotImplementedError, match="serves -tr nnUNetTrainerV2 \\| nnUNetTrainerV2BraTSRegions -m 3d_fullres"):
            NP.main(base + ["-tr", name])
    with pytest.raises(NotImplementedError, match="--save_softmax .* no background output"):
        NP.main(base + ["-tr", "nnUNetTrainerV2BraTSRegions", "--save_softmax"])
    assert not (tmp_path / "o").exists()
    # the region trainer's folder is found by its own name: a missing checkpoint is reported at that path
    os.remove(os.path.join(root, "nnUNet", "3d_fullres", "Task001_BrainTumour", "nnUNetTrainerV2BraTSRegions__nnUNetPlansv2.1",
                           "all", "model_best.model"))
    with pytest.raises(RuntimeError, match="nnUNetTrainerV2BraTSRegions__nnUNetPlansv2.1.*model_best.model"):
        NP.main(base + ["-tr", "nnUNetTrainerV2BraTSRegions"])
