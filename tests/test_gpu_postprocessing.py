"""nnU-Net v1 postprocessing.json on the device (dwmh_keep_largest_components, DESIGN §11), held bit for bit to the
restatement of upstream's remove_all_but_the_largest_connected_component (tests/postprocessing_oracle.py):

  * seeded multi-class label maps (smooth blobs plus scattered voxels), odd shapes (Z not a multiple of 32, one-voxel
    slabs along each axis, 37x41x53) and a 512x512x320 map, for every entry kind: one class, a class set, a set followed by
    its members, classes the map does not hold, minima met exactly, and labels >= 32 in the map;
  * planted ties of the largest size; a repeat call is bit-identical; voxels outside the mask are never written;
  * nnUNet_predict end to end on a two-modality, three-class model with a postprocessing.json in its trainer folder.
"""
import gzip
import json
import os

import numpy as np
import pytest
import torch

import oracle as O
import postprocessing_oracle as PO
from conftest import small_plans
from deepwmh_b200 import postprocessing as PP
from postprocessing_oracle import label_map

pytestmark = pytest.mark.gpu

VPV_ANISO = float(np.prod(np.array([0.9, 0.9, 3.0], np.float32), dtype=np.float64))   # float32 pixdim, as read from a header


@pytest.fixture(scope="module")
def net():
    import deepwmh_b200
    tr = deepwmh_b200.nnUNetTrainerV2(small_plans(), device=0, max_batch=1)
    yield tr.network
    tr.network.close()


def device_apply(net, seg, fwc, vpv, mins=None):
    d = torch.from_numpy(np.ascontiguousarray(seg)).cuda()
    PP.remove_all_but_the_largest_connected_component(net, d, fwc, vpv, mins)
    return d.cpu().numpy()


ENTRIES = [
    ([1], None),
    ([2], None),
    ([[1, 2]], None),
    ([[1, 2], 1, 2], None),
    ([2, 1], None),
    ([(1, 2), 2], {(1, 2): 40.0, 2: 3.0}),
    ([1, 2], {1: 0.0, 2: -1.0}),
    ([5, [2, 7]], None),                        # classes the map does not hold select nothing
]
SHAPES = [(37, 41, 53), (24, 24, 24), (64, 80, 48), (1, 40, 50), (30, 1, 45), (17, 23, 1), (5, 7, 3), (2, 3, 70)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_matches_upstream_bit_for_bit(net, shape):
    for seed in range(3):
        seg = label_map(shape, seed)
        for fwc, mins in ENTRIES:
            for vpv in (1.0, VPV_ANISO):
                got = device_apply(net, seg, fwc, vpv, mins)
                ref = PO.remove_all_but_the_largest_connected_component(seg, fwc, vpv, mins)
                assert np.array_equal(got, ref), (shape, seed, fwc, mins, vpv, int((got != ref).sum()))


def test_minimum_met_exactly_and_just_missed(net):
    """Minima equal to a component's fp64 size keep it; the next representable value above removes it."""
    from scipy.ndimage import label
    seg = label_map((40, 44, 36), 7)
    lmap, n = label(seg == 1)
    counts = np.bincount(lmap.ravel())[1:]
    assert n > 3
    for count in sorted(set(counts.tolist()))[:-1][-3:]:
        m = count * VPV_ANISO
        for mn in (m, np.nextafter(m, np.inf), np.nextafter(m, -np.inf)):
            got = device_apply(net, seg, [1], VPV_ANISO, {1: float(mn)})
            ref = PO.remove_all_but_the_largest_connected_component(seg, [1], VPV_ANISO, {1: float(mn)})
            assert np.array_equal(got, ref), (count, mn)


def test_planted_ties_keep_every_largest_component(net):
    seg = np.zeros((48, 50, 52), np.uint8)
    seg[2:7, 2:7, 2:7] = 1                      # 125 voxels
    seg[20:25, 30:35, 40:45] = 1                # 125 voxels
    seg[40:45, 5:10, 5:10] = 2                  # 125 voxels of class 2, for the class-set entry
    seg[30:32, 10:12, 10:12] = 1                # 8 voxels
    seg[10:11, 40:47, 0:1] = 2                  # 7 voxels
    for fwc in ([1], [[1, 2]], [2, 1]):
        got = device_apply(net, seg, fwc, 1.0)
        ref = PO.remove_all_but_the_largest_connected_component(seg, fwc, 1.0)
        assert np.array_equal(got, ref), fwc
    got = device_apply(net, seg, [1], 1.0)
    assert (got == 1).sum() == 250 and (got == 2).sum() == 132
    got = device_apply(net, seg, [[1, 2]], 1.0)
    assert (got == 1).sum() == 250 and (got == 2).sum() == 125


def test_labels_above_31_and_other_classes_are_never_written(net):
    rng = np.random.default_rng(2)
    seg = rng.integers(0, 256, size=(33, 35, 37), dtype=np.uint8)
    seg[rng.random(seg.shape) < 0.5] = 1
    for fwc in ([1], [[1, 31]], [31, 1]):
        got = device_apply(net, seg, fwc, 0.5)
        ref = PO.remove_all_but_the_largest_connected_component(seg, fwc, 0.5)
        assert np.array_equal(got, ref), fwc
        classes = set(np.ravel(fwc).tolist())
        untouched = ~np.isin(seg, list(classes))
        assert np.array_equal(got[untouched], seg[untouched])


def test_repeat_call_is_bit_identical_and_reuses_the_workspace(net):
    seg = label_map((64, 72, 40), 5, num_classes=4)
    fwc, mins = [[1, 2, 3], 3, 1], {(1, 2, 3): 10.0, 3: 4.0, 1: 2.0}
    a = device_apply(net, seg, fwc, VPV_ANISO, mins)
    small = label_map((9, 9, 9), 6)
    device_apply(net, small, [1], 1.0)          # a smaller map in between
    b = device_apply(net, seg, fwc, VPV_ANISO, mins)
    assert np.array_equal(a, b)
    assert np.array_equal(a, PO.remove_all_but_the_largest_connected_component(seg, fwc, VPV_ANISO, mins))


def test_large_map_512x512x320(net):
    seg = label_map((512, 512, 320), 9, sigma=2.0, scatter=0.001)
    for fwc in ([1], [[1, 2], 1, 2]):
        got = device_apply(net, seg, fwc, VPV_ANISO)
        ref = PO.remove_all_but_the_largest_connected_component(seg, fwc, VPV_ANISO)
        assert np.array_equal(got, ref), (fwc, int((got != ref).sum()))


def test_nnunet_predict_applies_postprocessing_json(tmp_path, monkeypatch, capsys):
    """T1 + FLAIR, three classes: the label file is upstream's postprocessing of the same run's --disable_post_processing
    output; the json is copied; without a json the output equals the flag's and the warning is printed; the softmax file is
    the same either way."""
    from deepwmh_b200 import nifti, nnunet_predict as NP
    from test_resample import _make_model_dir
    M, C = 2, 3
    plans = small_plans()
    plans["num_modalities"], plans["num_classes"] = M, C - 1
    plans["normalization_schemes"] = {m: "nonCT" for m in range(M)}
    plans["use_mask_for_norm"] = {m: True for m in range(M)}
    plans["plans_per_stage"][0]["current_spacing"] = np.array([1.2, 1.0, 1.0])
    net = O.build_benchmark_network(3, plans)
    root = str(tmp_path / "model")
    tdir = _make_model_dir(root, plans, net)
    indir = tmp_path / "in"; indir.mkdir()
    hdr = nifti.default_header((40, 44, 30), spacing=(1.0, 1.0, 1.1))
    for m in range(M):
        v = np.zeros((30, 44, 40), np.float32)
        v[2:28, 3:41, 4:37] = O.synthetic_flair((26, 38, 33), seed=40 + m)[0] * (1.0 + 0.5 * m)
        nifti.write_nifti(str(indir / ("caseB_%04d.nii.gz" % m)), np.transpose(v, (2, 1, 0)), hdr)
    monkeypatch.setenv("RESULTS_FOLDER", root)
    base = ["-i", str(indir), "-t", "Task002_FinalModel", "-f", "all", "-chk", "model_best", "--save_softmax"]

    def run(out, *extra):
        assert NP.main(base + ["-o", str(tmp_path / out)] + list(extra)) == 0
        return (nifti.read_nifti(str(tmp_path / out / "caseB.nii.gz")),
                gzip.open(str(tmp_path / out / "caseB.nii.gz")).read(), gzip.open(str(tmp_path / out / "caseB_0.nii.gz")).read())

    (raw_seg, raw_hdr), raw_bytes, raw_sm = run("off", "--disable_post_processing")
    pp = {"for_which_classes": [[1, 2], 1, 2], "dc_per_class_raw": {}, "dc_per_class_pp_final": {}}
    with open(os.path.join(tdir, "postprocessing.json"), "w") as f:
        json.dump(pp, f)
    (pp_seg, _), _, pp_sm = run("on")
    vpv = float(np.prod(np.asarray(raw_hdr["spacing"], dtype=np.float64)))
    ref = PO.remove_all_but_the_largest_connected_component(raw_seg, [(1, 2), 1, 2], vpv)
    print("postprocessing changed %d of %d voxels; labels %s" % (int((ref != raw_seg).sum()), raw_seg.size, np.unique(raw_seg)))
    assert np.array_equal(pp_seg, ref)
    assert (ref != raw_seg).any(), "the json removed nothing: the end-to-end case does not exercise it"
    assert json.load(open(tmp_path / "on" / "postprocessing.json")) == pp
    assert pp_sm == raw_sm
    assert not os.path.exists(tmp_path / "off" / "postprocessing.json")
    # with minima: written in upstream's str(dict) form
    with open(os.path.join(tdir, "postprocessing.json"), "w") as f:
        json.dump({"for_which_classes": [[1, 2], 2], "min_valid_object_sizes": str({(1, 2): 5.0, 2: 2.0})}, f)
    (mn_seg, _), _, _ = run("min")
    assert np.array_equal(mn_seg, PO.remove_all_but_the_largest_connected_component(raw_seg, [(1, 2), 2], vpv, {(1, 2): 5.0, 2: 2.0}))
    # no json: upstream's warning, and the same bytes as with the flag
    os.remove(os.path.join(tdir, "postprocessing.json"))
    capsys.readouterr()
    (_, _), none_bytes, none_sm = run("none")
    assert "Cannot run postprocessing because the postprocessing file is missing" in capsys.readouterr().out
    assert none_bytes == raw_bytes and none_sm == raw_sm
    assert not os.path.exists(tmp_path / "none" / "postprocessing.json")
