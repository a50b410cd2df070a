"""CPU restatement of nnU-Net v1's postprocessing, marked [U] like oracle/nnunet_oracle.py: recalled from upstream, not
diffed against it (the fork is not installed).  The device path (deepwmh_b200/postprocessing.py) is held to it bit for bit.

[U:postprocessing/connected_components.py::remove_all_but_the_largest_connected_component] with scipy.ndimage.label's
default structure (6-connectivity in 3-D); [U:postprocessing/connected_components.py::load_remove_save] computes
volume_per_voxel = prod(spacing of the written image) in fp64.  Upstream sizes each component with `(lmap == i).sum()` in
a loop; np.bincount gives the same counts in one pass, which keeps 512x512x320 maps affordable.
"""
import numpy as np
from scipy.ndimage import gaussian_filter, label


def remove_all_but_the_largest_connected_component(image, for_which_classes, volume_per_voxel, minimum_valid_object_size=None):
    image = np.array(image, copy=True)
    assert 0 not in for_which_classes, "cannot remove background"
    for c in for_which_classes:                               # in order; each entry sees what the previous ones left
        if isinstance(c, (list, tuple)):
            c = tuple(c)                                      # the key of minimum_valid_object_size
            assert 0 not in c, "cannot remove background"
            mask = np.isin(image, c)
        else:
            mask = image == c
        lmap, num_objects = label(mask.astype(int))
        if num_objects == 0:
            continue
        object_sizes = np.bincount(lmap.ravel(), minlength=num_objects + 1)[1:] * volume_per_voxel     # fp64, id 1..n
        maximum_size = object_sizes.max()
        remove = object_sizes != maximum_size                  # every component of the maximum size is kept
        if minimum_valid_object_size is not None:
            remove &= object_sizes < minimum_valid_object_size[c]
        image[np.concatenate([[False], remove])[lmap] & mask] = 0
    return image


def label_map(shape, seed, num_classes=3, sigma=1.5, scatter=0.02):
    """Seeded test input: smooth blobs of classes 1 .. C-1 on background, plus a fraction `scatter` of voxels set to random
    classes (many small components next to a few large ones)."""
    rng = np.random.default_rng(seed)
    f = gaussian_filter(rng.standard_normal(shape, dtype=np.float32), sigma=min(sigma, max(shape) / 4), mode="wrap")
    q = np.quantile(f, np.linspace(0.45, 1.0, num_classes)[:-1])
    seg = np.digitize(f, q).astype(np.uint8)
    pick = rng.random(shape) < scatter
    seg[pick] = rng.integers(0, num_classes, size=int(pick.sum()), dtype=np.uint8)
    return seg
