"""oracle/intree_oracle.py against tests/golden/intree_v1.npz -- outputs of the REFERENCE'S OWN functions
(deepwmh/analysis/image_ops.py, lesion_analysis.py, metrics.py, pipeline/DCNN_multistage.py) run by
tests/golden/make_golden_intree.py (read through tests/golden/fixtures.py: volumes compared with a tolerance are held
on a fixed voxel sample, `g.sample`).  These rows of SURVEY.md section 8 (a2 sibling z_score, f-2, f-3, f-4) are
therefore pinned; the nnU-Net engine rows stay `parity unpinned` (oracle/__init__.py)."""
import numpy as np
import pytest

from oracle import intree_oracle as I
from deepwmh_b200 import preprocess
from golden import fixtures as F

# volumes in the fixture are stored as float32: one rounding of the reference's float64 result
F32 = dict(rtol=2e-6, atol=2e-6)


@pytest.fixture(scope="module")
def g():
    return F.intree()


def test_fixture_was_made_by_the_reference(g):
    assert "nibabel" in set(g["stubbed_modules"].tolist())          # absent third-party modules were stand-ins only
    assert str(g["ens_y0_dtype"]) == "float32"


def test_z_score_and_masked_stats(g):
    mn, sd = I.masked_mean_std(g["in_target"], g["in_brain"])
    assert np.allclose([mn, sd], g["masked_mean_std"], rtol=1e-6)   # the reference sums in float32 here
    assert np.allclose(I.z_score(g["in_target"], g["in_brain"]), g["zscore_masked"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(I.z_score(g["in_target"])), g["zscore_plain"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("tag", ["iso1", "iso05", "iso2", "thick", "aniso"])
def test_remove_3mm_sparks(g, tag):
    vox = g["sparks_vox_" + tag].tolist()
    assert np.array_equal(I.remove_3mm_sparks(g["sparks_in"], vox), g["sparks_" + tag])
    assert np.array_equal(preprocess.remove_3mm_sparks(g["sparks_in"], vox), g["sparks_" + tag])   # host rule of the product
    assert g["sparks_" + tag].sum() < (g["sparks_in"] > 0.5).sum()


def test_remove_sparks_min_volume(g):
    assert np.array_equal(I.remove_sparks(g["sparks_in"], 5), g["sparks_min5"])


def test_stage2_masking_and_ensembling_bit_exact(g):
    masked = [I.softmax_masking(x, g["ens_mask"]) for x in g["ens_x"]]
    field, lab = I.ensembling(masked, [1.0, 1.0, 1.0])
    assert field.dtype == np.float32 and np.array_equal(field, g["ens_field"])
    assert np.array_equal(lab, g["ens_label"])


def test_hard_dice(g):
    names = g["dice_names"].tolist()
    ref = g["dice_vals"][names.index("hard_dice_binary")]
    assert I.hard_dice_binary(g["dice_in"][0], g["dice_in"][1]) == pytest.approx(ref, rel=1e-7)   # fp32 sums in the reference


def test_the_parity_gates_own_helpers_are_pinned_too(g):
    """oracle/nnunet_oracle.py: the Dice the BASELINE gate is quoted in and the in-tree z_score sibling, against the reference's output."""
    import oracle as O
    names = g["dice_names"].tolist()
    ref = g["dice_vals"][names.index("hard_dice_binary")]
    assert O.hard_dice_binary(g["dice_in"][0], g["dice_in"][1]) == pytest.approx(ref, rel=1e-7)
    assert np.allclose(O.zscore_deepwmh(g["in_target"], g["in_brain"]), g["zscore_masked"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(O.zscore_deepwmh(g["in_target"])), g["zscore_plain"], rtol=1e-5, atol=1e-5)


def test_group_statistics_and_nll(g):
    zt, zr = g["z_target"], list(g["z_refs"])
    assert np.allclose(g.sample(I.group_mean(zr)), g["group_mean"], **F32)
    assert np.allclose(g.sample(I.group_std(zr)), g["group_std"], **F32)
    for side, tag in ((None, "none"), ("+", "pos"), ("-", "neg")):
        an, mu, sg = I.nll(zt, zr, min_std=0.03, side=side, return_all=True)
        assert np.allclose(an if tag == "pos" else g.sample(an), g["nll_" + tag], **F32)
    assert np.allclose(g.sample(mu), g["nll_mu"], **F32) and np.allclose(g.sample(sg), g["nll_sigma"], **F32)
    assert np.allclose(g.sample(I.nll(zt, zr)), g["nll_eps"], **F32)
    assert (g.sample(g["nll_pos"]) != g["nll_none"]).any() and (g["nll_sigma"] >= np.float32(0.03)).all()


def test_masked_group_statistics_and_otsu_branch_of_nll(g):
    zt, zr, gm = g["z_target"], list(g["z_refs"]), list(g["gmask"])
    assert np.allclose(g.sample(I.group_mean(zr, gm)), g["group_mean_masked"], equal_nan=True, **F32)
    assert np.allclose(g.sample(I.group_std(zr, gm)), g["group_std_masked"], equal_nan=True, **F32)
    slab = np.zeros(zt.shape, bool)
    slab[5:9] = True
    assert np.isnan(g["group_mean_masked"][g.sample(slab)]).all()
    assert np.array_equal(np.isnan(g["group_mean_masked"]), g.sample((np.stack(gm) < 0.5).all(axis=0)))     # NaN exactly where nothing is left
    an, mu, sg = I.nll(zt, zr, min_std=0.03, side="+", return_all=True, use_mask=True)     # reference code + restated Otsu
    assert np.allclose(g.sample(an), g["nll_usemask"], **F32) and np.allclose(g.sample(mu), g["nll_usemask_mu"], equal_nan=True, **F32)
    assert np.allclose(g.sample(sg), g["nll_usemask_sigma"], equal_nan=True, **F32)


@pytest.mark.parametrize("tag", ["p12", "p50", "podd", "nomask"])
def test_mean_std_grid(g, tag):
    if tag == "nomask":
        m, s = I.mean_std_grid(g["z_target"], [12, 12, 12])
    else:
        m, s = I.mean_std_grid(g["z_target"], g["msg_patch_" + tag].tolist(), mask=g["in_valid"])
    assert m.shape == g["z_target"].shape
    assert np.allclose(g.sample(m), g["msg_mean_" + tag], rtol=1e-5, atol=1e-6)
    assert np.allclose(g.sample(s), g["msg_std_" + tag], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("tag,ks", [("iso1", [3, 3, 3]), ("iso07", [4, 4, 4]), ("mixed", [6, 5, 3]), ("thick", [3, 3, 1])])
def test_median_3mm(g, tag, ks):
    vox = g["median_vox_" + tag].tolist()
    assert I.median_kernel(vox) == ks
    assert np.array_equal(I.median_3mm(g["nll_pos"], vox), g["median_" + tag])


@pytest.mark.parametrize("tag", ["iso", "thick_z", "thick_x"])
def test_component_filtering(g, tag):
    assert np.array_equal(I.component_filtering(g["cf_in"], g["cf_vox_" + tag].tolist()), g["cf_" + tag])


def test_component_filtering_edge_cases(g):
    assert np.array_equal(I.component_filtering(g["in_brain"], [1.0, 1.0, 1.0]), g["cf_brain"])
    assert np.array_equal(I.component_filtering(np.zeros((6, 7, 5), np.float32), [1.0, 1.0, 1.0]), g["cf_empty"])
    assert g["cf_iso"].sum() < g["cf_in"].sum() and g["cf_iso"][2:4, 3:6, 4:6].sum() == 0      # the sparks are gone
    assert np.array_equal(g["cf_thick_z"], g["cf_in"])             # thick slices: two orientations pass the mask through


def test_anomaly_pipeline(g):
    r = I.nll_anomaly_arrays(g["in_target"], list(g["in_refs"]), g["in_brain"], g["in_valid"], g["pipe_patch"].tolist())
    assert np.allclose(g.sample(r["x_prime"]), g["pipe_x_prime"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(r["local_mu"]), g["pipe_local_mu"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(r["mean"]), g["pipe_mean"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(r["std"]), g["pipe_std"], rtol=1e-4, atol=1e-5)
    # (x - mu)^2 / (2 sigma^2) with sigma floored at 0.03 magnifies 1e-7 input differences ~1e3-fold
    assert np.allclose(g.sample(r["anomaly"]), g["pipe_anomaly"], rtol=1e-4, atol=2e-3)
    an0 = I.nll(r["refs"][0], r["refs"], min_std=0.03, side="+") * g["in_valid"]
    assert np.allclose(g.sample(an0), g["pipe_ref_anomaly0"], rtol=1e-4, atol=2e-3)


@pytest.mark.parametrize("tag,prior", [("pos", "+"), ("none", None)])
def test_whole_nll_analysis_against_the_reference_run_end_to_end(tag, prior):
    """tests/golden/nll_analysis_v1.npz = the reference's nll_analysis itself (NIfTI I/O redirected to memory)."""
    f = F.nll_analysis()
    an, valid, cx, cy, cr, thr, ex = I.nll_analysis_arrays(f["in_target"], list(f["in_refs"]), list(f["in_label1"]),
                                                           [t.astype(np.float32) for t in f["in_label2"]], f["voxel_size"].tolist(), prior)
    assert np.array_equal(valid, f["valid_" + tag]) and np.array_equal(ex["rough_brain"], f["rough_brain_" + tag])
    assert np.array_equal(ex["averaged_label"], f["averaged_label_" + tag])
    assert np.allclose(f.sample(ex["x_prime"]), f["normalized_input_" + tag], rtol=1e-5, atol=1e-5)
    assert np.allclose(f.sample(ex["mean"]), f["mean_value_" + tag], rtol=1e-5, atol=1e-5)
    assert np.allclose(an, f["anomaly_" + tag], rtol=1e-4, atol=2e-3)
    assert np.allclose(cx, f["curve_x_" + tag], rtol=1e-6) and np.allclose(cy, f["curve_y_" + tag], atol=1e-6)
    assert np.allclose(cr, f["curve_r_" + tag], atol=1e-6) and thr == pytest.approx(float(f["threshold_" + tag]), rel=1e-6)
    assert an[20:23, 12:15, 6:9].max() > thr and an[14:18, 22:27, 20:24].max() > thr      # both planted lesions are found
