"""nnU-Net v1 postprocessing (`postprocessing.json` in the trainer folder) on the device, DESIGN §11.

[U:postprocessing/connected_components.py]: for each entry of `for_which_classes`, in order and on the label map as the
previous entries left it, every 6-connected component of the entry's class set is set to 0 except the largest ones (ties
are all kept) and, when `min_valid_object_sizes` is given, except those of at least that many mm^3.  An entry is one
class id or a list of ids that count as one foreground.  Same function names and json format as upstream; the component
labelling and the filter are `dwmh_keep_largest_components` (deepwmh_b200/csrc/kernels_ccl.cuh).
"""
from __future__ import annotations

import ast
import json
import numbers
from typing import Dict, List, Optional, Tuple, Union

Entry = Union[int, Tuple[int, ...]]

MAX_CLASS_ID = 31          # the class set travels as a 32-bit mask


def _key(entry) -> Entry:
    """The entry as upstream looks it up in min_valid_object_sizes: an int, or a tuple for a list of classes."""
    return tuple(entry) if isinstance(entry, (list, tuple)) else entry


def class_mask(entry) -> int:
    """Bit c set for every class c of the entry; raises ValueError for anything upstream would not treat as class ids
    (and for ids above 31).  Class 0 is refused as upstream asserts: the background cannot be removed."""
    classes = list(entry) if isinstance(entry, (list, tuple)) else [entry]
    if not classes:
        raise ValueError("postprocessing entry %r selects no class" % (entry,))
    mask = 0
    for c in classes:
        if isinstance(c, bool) or not isinstance(c, numbers.Integral):
            raise ValueError("postprocessing entry %r: class id %r is not an int" % (entry, c))
        if c == 0:
            raise ValueError("postprocessing entry %r: cannot remove background (class 0)" % (entry,))
        if c < 0 or c > MAX_CLASS_ID:
            raise ValueError("postprocessing entry %r: class id %d outside 1..%d" % (entry, c, MAX_CLASS_ID))
        mask |= 1 << int(c)
    return mask


def load_postprocessing(json_file: str) -> Tuple[List[Entry], Optional[Dict]]:
    """[U:postprocessing/connected_components.py::load_postprocessing] -> (for_which_classes, min_valid_object_sizes).
    Entries come back as ints and tuples; min_valid_object_sizes is `ast.literal_eval` of the json string, or None when the
    key is absent.  Everything the device call would refuse, and a minimum missing for one of the entries, raises here."""
    with open(json_file) as f:
        a = json.load(f)
    if not isinstance(a, dict) or not isinstance(a.get("for_which_classes"), list):
        raise ValueError("%s: expected an object with a for_which_classes list" % json_file)
    entries = [_key(e) for e in a["for_which_classes"]]
    for e in entries:
        class_mask(e)
    min_sizes = None
    if "min_valid_object_sizes" in a:
        raw = a["min_valid_object_sizes"]
        if not isinstance(raw, str):
            raise ValueError("%s: min_valid_object_sizes must be the string form of a dict, got %r" % (json_file, raw))
        min_sizes = ast.literal_eval(raw)
        if not isinstance(min_sizes, dict):
            raise ValueError("%s: min_valid_object_sizes is not a dict: %r" % (json_file, raw))
        for e in entries:
            if e not in min_sizes:
                raise ValueError("%s: min_valid_object_sizes has no entry for %r" % (json_file, e))
            v = min_sizes[e]
            if isinstance(v, bool) or not isinstance(v, numbers.Real):
                raise ValueError("%s: min_valid_object_sizes[%r] = %r is not a number" % (json_file, e, v))
    return entries, min_sizes


def remove_all_but_the_largest_connected_component(network, seg_dev, for_which_classes, volume_per_voxel: float,
                                                   minimum_valid_object_size: Optional[Dict] = None):
    """[U:postprocessing/connected_components.py::remove_all_but_the_largest_connected_component] in place on a
    contiguous uint8 CUDA label map: one device call per entry, in order.  volume_per_voxel: the product of the written
    image's spacing in fp64.  Returns seg_dev."""
    for entry in for_which_classes:
        mask = class_mask(entry)
        min_mm3 = -1.0                                          # < 0: no minimum, only the largest components stay
        if minimum_valid_object_size is not None:
            m = float(minimum_valid_object_size[_key(entry)])
            # upstream removes a component iff its size < m: for m <= 0 or NaN nothing is removed, which a minimum of 0 says too
            min_mm3 = m if m >= 0.0 else 0.0
        network.keep_largest_components_(seg_dev, mask, volume_per_voxel, min_mm3)
    return seg_dev
