"""Host-side logic of deepwmh_b200/stage1.py (no GPU): kernel-size / patch-size rules, the Otsu scan and the threshold
search, against the reference-pinned oracle (oracle/intree_oracle.py) and the reference's own end-to-end output."""
import numpy as np
import pytest

from oracle import intree_oracle as I
from deepwmh_b200 import stage1 as S
from golden import fixtures as F


@pytest.mark.parametrize("vox", [[1, 1, 1], [0.7, 0.7, 0.7], [0.5, 0.6, 1.5], [0.9, 0.9, 5.0], [6.0, 1.0, 1.0], [0.4, 3.0, 0.4], [2, 2, 2]])
def test_median_kernel_rule(vox):
    assert S.median_kernel_size(vox) == I.median_kernel(vox)


def test_median_kernel_rule_matches_reference_fixture():
    g = F.intree()
    for tag, ks in (("iso1", [3, 3, 3]), ("iso07", [4, 4, 4]), ("mixed", [6, 5, 3]), ("thick", [3, 3, 1])):
        assert S.median_kernel_size(g["median_vox_" + tag].tolist()) == ks


def test_image_patch_size():
    assert S.image_patch_size([1.0, 1.2, 1.1]) == [50, 42, 46]        # what the reference printed for the fixture case
    assert S.image_patch_size([0.5, 0.5, 5.0]) == [100, 100, 10]


def test_otsu_scan_equals_the_restatement():
    rng = np.random.default_rng(0)
    for _ in range(5):
        v = np.concatenate([rng.normal(0, 1, 5000), rng.normal(rng.uniform(2, 6), 0.7, 3000)])
        counts, edges = np.histogram(v, bins=256)
        assert S._otsu_from_histogram(counts, edges) == I.threshold_otsu(v)
    counts, edges = np.histogram(np.array([0.0, 0.0, 1.0, 1.0]), bins=256)     # empty bins: divisions by zero are ignored
    assert S._otsu_from_histogram(counts, edges) == I.threshold_otsu(np.array([0.0, 0.0, 1.0, 1.0]))


def test_threshold_search_on_the_reference_curves():
    f = F.nll_analysis()
    for tag, prior in (("pos", "+"), ("none", None)):
        _, _, cx, _, _, thr, _ = I.nll_analysis_arrays(f["in_target"], list(f["in_refs"]), list(f["in_label1"]),
                                                       [t.astype(np.float32) for t in f["in_label2"]], f["voxel_size"].tolist(), prior)
        assert thr == pytest.approx(float(f["threshold_" + tag]), rel=1e-6)
    # synthetic curves: right-most bin above 0.01 per reference, median over references
    x = np.arange(10, dtype=np.float64) + 0.5
    rs = [np.array([5, 4, 3, 0.3, 0, 0, 0, 0, 0, 0.0]), np.array([5, 4, 3, 2, 1, 0.3, 0, 0, 0, 0.0]), np.array([5, 0, 0, 0, 0, 0, 0, 0.3, 0, 0.0])]
    assert S.anomaly_threshold_from_curves(x, rs) == 5.5
    assert S._side(None) == 0 and S._side("+") == 1 and S._side("-") == -1
    with pytest.raises(AssertionError):
        S._side("both")


def test_unsupported_branches_raise_without_a_gpu():
    z = np.zeros((4, 4, 4), np.float32)
    with pytest.raises(NotImplementedError):
        S.mean_std_grid(z, [2, 2, 2], order=3)
    with pytest.raises(NotImplementedError):
        S.component_filtering(z, [1, 1, 1], return_type="int")
