"""CPU: nnU-Net v1 postprocessing.json (keep the largest connected component, DESIGN §11).

  * known answers of the upstream restatement (tests/postprocessing_oracle.py) that the device path is held to;
  * load_postprocessing on tuple keys, an absent min_valid_object_sizes, an empty list and every rejection;
  * the argument checks of dwmh_keep_largest_components through the C ABI (no device or context needed);
  * nnUNet_predict refuses a malformed postprocessing.json before any GPU work.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import postprocessing_oracle as PO
from deepwmh_b200 import _lib, postprocessing as PP


def _box(img, lo, hi, v):
    img[tuple(slice(a, b) for a, b in zip(lo, hi))] = v


# ---- known answers of the restatement -------------------------------------------------------------------------------

def test_two_equal_largest_components_are_both_kept():
    img = np.zeros((10, 10, 10), np.uint8)
    _box(img, (0, 0, 0), (2, 2, 2), 1)          # 8 voxels
    _box(img, (5, 5, 5), (7, 7, 7), 1)          # 8 voxels
    _box(img, (9, 0, 0), (10, 1, 2), 1)         # 2 voxels
    out = PO.remove_all_but_the_largest_connected_component(img, [1], 1.0)
    assert (out == 1).sum() == 16 and out[9, 0, 0] == 0


def test_minimum_size_keeps_components_at_or_above_it():
    img = np.zeros((12, 12, 12), np.uint8)
    _box(img, (0, 0, 0), (3, 3, 3), 1)          # 27 voxels: the largest
    _box(img, (6, 6, 6), (8, 8, 8), 1)          # 8 voxels
    _box(img, (10, 0, 0), (11, 1, 3), 1)        # 3 voxels
    vpv = 0.5                                   # 8 voxels = 4 mm^3, 3 voxels = 1.5 mm^3
    out = PO.remove_all_but_the_largest_connected_component(img, [1], vpv, {1: 4.0})
    assert (out == 1).sum() == 35               # 4.0 >= 4.0 is kept; 1.5 < 4.0 is removed
    out = PO.remove_all_but_the_largest_connected_component(img, [1], vpv, {1: 4.0000001})
    assert (out == 1).sum() == 27


def test_tuple_entry_merges_touching_classes():
    img = np.zeros((10, 10, 10), np.uint8)
    _box(img, (0, 0, 0), (2, 2, 2), 1)
    _box(img, (2, 0, 0), (4, 2, 2), 2)          # touches the class-1 box: one 16-voxel component of {1, 2}
    _box(img, (6, 6, 6), (9, 9, 9), 1)          # 27 voxels of class 1 alone
    alone = PO.remove_all_but_the_largest_connected_component(img, [1], 1.0)
    assert (alone == 1).sum() == 27 and (alone == 2).sum() == 8
    merged = PO.remove_all_but_the_largest_connected_component(img, [(1, 2)], 1.0)
    assert (merged == 1).sum() == 27 and (merged == 2).sum() == 0          # the 16-voxel {1, 2} component goes as one
    _box(img, (4, 0, 0), (6, 4, 4), 2)          # now the {1, 2} component (48 voxels) is the largest
    merged = PO.remove_all_but_the_largest_connected_component(img, [[1, 2]], 1.0)
    assert (merged == 1).sum() == 8 and (merged == 2).sum() == 40
    assert (merged[6:9, 6:9, 6:9] == 0).all()


def test_entry_order_matters():
    """[1, 2] then 1 differs from 1 alone: the merged entry first removes a class-1 component that would be the largest of
    class 1, so the second entry keeps a different one."""
    img = np.zeros((12, 12, 12), np.uint8)
    _box(img, (0, 0, 0), (3, 3, 3), 1)          # A: 27 voxels of class 1, isolated
    _box(img, (6, 6, 6), (8, 8, 8), 1)          # B: 8 voxels of class 1 ...
    _box(img, (8, 6, 6), (12, 12, 12), 2)       # ... touching 144 voxels of class 2: B + class 2 is the largest {1, 2} component
    one = PO.remove_all_but_the_largest_connected_component(img, [1], 1.0)
    both = PO.remove_all_but_the_largest_connected_component(img, [[1, 2], 1], 1.0)
    assert (one[0:3, 0:3, 0:3] == 1).all() and (one[6:8, 6:8, 6:8] == 0).all()
    assert (both[0:3, 0:3, 0:3] == 0).all() and (both[6:8, 6:8, 6:8] == 1).all() and (both == 2).sum() == 144


def test_single_class_entry_does_not_connect_through_another_class():
    img = np.zeros((3, 3, 9), np.uint8)
    img[1, 1, 0:3] = 1
    img[1, 1, 3] = 2                            # a class-2 bridge
    img[1, 1, 4:6] = 1
    out = PO.remove_all_but_the_largest_connected_component(img, [1], 1.0)
    assert out[1, 1, 0:3].tolist() == [1, 1, 1] and out[1, 1, 3] == 2 and out[1, 1, 4:6].tolist() == [0, 0]
    out = PO.remove_all_but_the_largest_connected_component(img, [(1, 2)], 1.0)
    assert np.array_equal(out, img)             # through the bridge it is one component


def test_diagonal_neighbours_are_separate_components():
    img = np.zeros((4, 4, 4), np.uint8)
    img[0, 0, 0:2] = 1
    img[1, 1, 2] = 1                            # touches only along an edge: not 6-connected
    out = PO.remove_all_but_the_largest_connected_component(img, [1], 1.0)
    assert out[1, 1, 2] == 0 and out.sum() == 2


def test_class_zero_raises():
    img = np.ones((2, 2, 2), np.uint8)
    with pytest.raises(AssertionError):
        PO.remove_all_but_the_largest_connected_component(img, [0], 1.0)
    with pytest.raises(AssertionError):
        PO.remove_all_but_the_largest_connected_component(img, [[0, 1]], 1.0)
    with pytest.raises(ValueError):
        PP.class_mask(0)
    with pytest.raises(ValueError):
        PP.class_mask([1, 0])


# ---- load_postprocessing --------------------------------------------------------------------------------------------

def _json(tmp_path, obj, name="postprocessing.json"):
    p = tmp_path / name
    p.write_text(json.dumps(obj))
    return str(p)


def test_load_tuple_keys_and_min_sizes(tmp_path):
    # the form upstream's determine_postprocessing writes: lists in for_which_classes, str(dict) with tuple keys
    p = _json(tmp_path, {"for_which_classes": [[1, 2], 1, 2], "min_valid_object_sizes": "{(1, 2): 120.0, 1: 30.0, 2: 7}",
                         "dc_per_class_raw": {"1": 0.8}})
    fwc, mins = PP.load_postprocessing(p)
    assert fwc == [(1, 2), 1, 2] and mins == {(1, 2): 120.0, 1: 30.0, 2: 7}
    assert [PP.class_mask(e) for e in fwc] == [0b110, 0b10, 0b100]


def test_load_without_min_sizes_and_empty_list(tmp_path):
    assert PP.load_postprocessing(_json(tmp_path, {"for_which_classes": [1, [2, 3]]})) == ([1, (2, 3)], None)
    assert PP.load_postprocessing(_json(tmp_path, {"for_which_classes": []})) == ([], None)
    assert PP.load_postprocessing(_json(tmp_path, {"for_which_classes": [], "min_valid_object_sizes": "{}"})) == ([], {})
    assert PP.class_mask(31) == 1 << 31           # the highest class id the 32-bit mask carries


@pytest.mark.parametrize("obj, what", [
    ({"for_which_classes": [0]}, "background"),
    ({"for_which_classes": [[1, 0]]}, "background"),
    ({"for_which_classes": [-1]}, "outside"),
    ({"for_which_classes": [32]}, "outside"),
    ({"for_which_classes": [1.0]}, "not an int"),
    ({"for_which_classes": ["1"]}, "not an int"),
    ({"for_which_classes": [True]}, "not an int"),
    ({"for_which_classes": [[1, [2]]]}, "not an int"),
    ({"for_which_classes": [[]]}, "no class"),
    ({"for_which_classes": 1}, "for_which_classes list"),
    ({}, "for_which_classes list"),
    ({"for_which_classes": [1, [1, 2]], "min_valid_object_sizes": "{1: 10.0}"}, "no entry for (1, 2)"),
    ({"for_which_classes": [[1, 2]], "min_valid_object_sizes": "{1: 10.0, 2: 3.0}"}, "no entry for (1, 2)"),
    ({"for_which_classes": [1], "min_valid_object_sizes": {"1": 10.0}}, "string form"),
    ({"for_which_classes": [1], "min_valid_object_sizes": "[1, 2]"}, "not a dict"),
    ({"for_which_classes": [1], "min_valid_object_sizes": "{1: 'a'}"}, "not a number"),
])
def test_load_rejects(tmp_path, obj, what):
    with pytest.raises(ValueError, match=what.replace("(", r"\(").replace(")", r"\)")):
        PP.load_postprocessing(_json(tmp_path, obj))


class _RecordingNetwork:
    def __init__(self):
        self.calls = []

    def keep_largest_components_(self, seg, class_mask, volume_per_voxel, min_valid_mm3=-1.0):
        self.calls.append((class_mask, volume_per_voxel, min_valid_mm3))
        return seg


def test_one_device_call_per_entry_in_order_with_its_minimum():
    net = _RecordingNetwork()
    mins = {(1, 2): 120.0, 1: 0.0, 2: -5.0, 3: float("nan"), 4: float("inf")}
    PP.remove_all_but_the_largest_connected_component(net, None, [[1, 2], 1, 2, 3, 4], 0.25, mins)
    # a minimum <= 0 or NaN removes nothing upstream (size < m is false for every size): the device is told 0
    assert net.calls == [(6, 0.25, 120.0), (2, 0.25, 0.0), (4, 0.25, 0.0), (8, 0.25, 0.0), (16, 0.25, float("inf"))]
    net = _RecordingNetwork()
    PP.remove_all_but_the_largest_connected_component(net, None, [3, (1, 3)], 1.5)
    assert net.calls == [(8, 1.5, -1.0), (10, 1.5, -1.0)]
    PP.remove_all_but_the_largest_connected_component(net, None, [], 1.5)
    assert len(net.calls) == 2


def _upstream_loop(image, for_which_classes, volume_per_voxel, minimum_valid_object_size=None):
    """The restatement's arithmetic written as upstream's per-component loop."""
    from scipy.ndimage import label
    image = np.array(image, copy=True)
    for c in for_which_classes:
        if isinstance(c, (list, tuple)):
            c = tuple(c)
            mask = np.zeros_like(image, dtype=bool)
            for cl in c:
                mask[image == cl] = True
        else:
            mask = image == c
        lmap, num_objects = label(mask.astype(int))
        object_sizes = {i: (lmap == i).sum() * volume_per_voxel for i in range(1, num_objects + 1)}
        if num_objects > 0:
            maximum_size = max(object_sizes.values())
            for i in range(1, num_objects + 1):
                if object_sizes[i] != maximum_size:
                    remove = True
                    if minimum_valid_object_size is not None:
                        remove = object_sizes[i] < minimum_valid_object_size[c]
                    if remove:
                        image[(lmap == i) & mask] = 0
    return image


@pytest.mark.parametrize("seed", range(4))
def test_restatement_equals_upstreams_per_component_loop(seed):
    rng = np.random.default_rng(seed)
    img = rng.choice(4, size=(9, 11, 13), p=[0.55, 0.2, 0.15, 0.1]).astype(np.uint8)
    vpv = float(np.prod(np.array([0.9, 0.9, 3.0], np.float32), dtype=np.float64))
    for fwc, mins in (([1], None), ([[1, 2], 1, 2], None), ([3, [1, 3]], {3: 2 * vpv, (1, 3): 5.0}), ([2, 1], {2: 0.0, 1: 1e9})):
        assert np.array_equal(PO.remove_all_but_the_largest_connected_component(img, fwc, vpv, mins),
                              _upstream_loop(img, fwc, vpv, mins)), (fwc, mins)


def test_restatement_agrees_with_a_minimum_of_zero_for_nonpositive_and_nan_minima():
    rng = np.random.default_rng(3)
    img = (rng.random((12, 13, 14)) < 0.3).astype(np.uint8)
    ref0 = PO.remove_all_but_the_largest_connected_component(img, [1], 0.7, {1: 0.0})
    assert np.array_equal(ref0, img)
    for m in (-3.0, float("nan"), float("-inf")):
        assert np.array_equal(PO.remove_all_but_the_largest_connected_component(img, [1], 0.7, {1: m}), ref0)


# ---- C ABI argument checks ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("args, msg", [
    ((0, 4, 4, 2, 1.0, -1.0), b"empty volume"),
    ((4, -1, 4, 2, 1.0, -1.0), b"empty volume"),
    ((2048, 1024, 1024, 2, 1.0, -1.0), b"exceeds the 32-bit label range"),
    ((4, 4, 4, 0, 1.0, -1.0), b"selects no class"),
    ((4, 4, 4, 3, 1.0, -1.0), b"cannot remove background"),
    ((4, 4, 4, 1, 1.0, -1.0), b"cannot remove background"),
    ((4, 4, 4, 2, 0.0, -1.0), b"volume_per_voxel"),
    ((4, 4, 4, 2, -1.0, -1.0), b"volume_per_voxel"),
    ((4, 4, 4, 2, float("inf"), -1.0), b"volume_per_voxel"),
    ((4, 4, 4, 2, float("nan"), -1.0), b"volume_per_voxel"),
    ((4, 4, 4, 2, 1.0, float("nan")), b"min_valid_mm3 is NaN"),
    ((4, 4, 4, 2, 1.0, -1.0), b"null argument"),
])
def test_entry_point_refuses_bad_arguments_before_any_device_work(args, msg):
    lib = _lib.load()
    X, Y, Z, mask, vpv, mn = args
    rc = lib.dwmh_keep_largest_components(None, None, X, Y, Z, mask, vpv, mn, None)
    assert rc != 0 and msg in lib.dwmh_last_error(), lib.dwmh_last_error()


# ---- nnUNet_predict --------------------------------------------------------------------------------------------------

def test_nnunet_predict_refuses_a_malformed_json_before_gpu_work(tmp_path, monkeypatch):
    import pickle
    from conftest import small_plans
    from deepwmh_b200 import nnunet_predict as NP
    tdir = tmp_path / "m" / "nnUNet" / "3d_fullres" / "Task002_FinalModel" / "nnUNetTrainerV2__nnUNetPlansv2.1"
    (tdir / "all").mkdir(parents=True)
    pickle.dump(small_plans(), open(tdir / "plans.pkl", "wb"))
    (tdir / "all" / "model_best.model").write_bytes(b"not read before the json is")
    (tdir / "postprocessing.json").write_text(json.dumps({"for_which_classes": [0]}))
    indir = tmp_path / "in"; indir.mkdir()
    (indir / "c_0000.nii.gz").write_bytes(b"")
    monkeypatch.setenv("RESULTS_FOLDER", str(tmp_path / "m"))
    out = tmp_path / "out"
    argv = ["-i", str(indir), "-o", str(out), "-t", "Task002_FinalModel", "-f", "all", "-chk", "model_best"]
    with pytest.raises(ValueError, match="background"):
        NP.main(argv)
    assert not out.exists()
