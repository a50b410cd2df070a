"""SURVEY.md section 8f-4 on the device: deepwmh_b200/stage1.py (dwmh_s1_* through the C ABI) against

  * tests/golden/intree_v1.npz -- outputs of the REFERENCE'S OWN functions (tests/golden/make_golden_intree.py; volumes
    compared with a tolerance are held on a fixed voxel sample, `g.sample`, see tests/golden/fixtures.py), and
  * oracle/intree_oracle.py on seeded inputs, at small sizes and at BASELINE.json's 182x218x182.

Tolerances: the device stores fp32 and computes each voxel in fp64; the reference computes in the dtype numpy promotes
to (float32 sums for float32 inputs in group_mean / group_std, float64 after z_score).  Integer / selection work (median
filter) is bit-exact.  The NLL magnifies input differences by (x - mu) / sigma^2 <= ~1e3 (sigma floored at 0.03), hence
rtol 1e-4 / atol 2e-3 where the inputs themselves come from the device z-score."""
import numpy as np
import pytest
import torch

from oracle import intree_oracle as I
from golden import fixtures as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def g():
    return F.intree()


@pytest.fixture(scope="module")
def S():
    from deepwmh_b200 import stage1
    return stage1


def h(t):
    return t.cpu().numpy()


def test_z_score_matches_reference_fixture(g, S):
    z, st = S.z_score(g["in_target"], g["in_brain"], return_stats=True)
    assert np.allclose(st[:2], g["masked_mean_std"], rtol=1e-6) and st[2] == (g["in_brain"] > 0.5).sum()
    assert np.allclose(h(z), g["zscore_masked"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(h(S.z_score(g["in_target"]))), g["zscore_plain"], rtol=1e-5, atol=1e-5)
    # input untouched, numpy or tensor
    t = torch.from_numpy(g["in_target"]).cuda()
    S.z_score(t, g["in_brain"])
    assert np.array_equal(h(t), g["in_target"])
    filled = h(S.z_score(g["in_target"], g["in_brain"], fill_outside=True))
    assert np.allclose(g.sample(filled), g["pipe_x_prime"], rtol=1e-5, atol=1e-5)
    with pytest.raises(Exception):
        S.z_score(g["in_target"], None, fill_outside=True)


def test_group_statistics_and_nll_match_reference_fixture(g, S):
    zt, zr = g["z_target"], list(g["z_refs"])
    assert np.allclose(g.sample(h(S.group_mean(zr))), g["group_mean"], rtol=1e-6, atol=1e-6)
    assert np.allclose(g.sample(h(S.group_std(zr))), g["group_std"], rtol=1e-5, atol=1e-6)
    for side, tag in ((None, "none"), ("+", "pos"), ("-", "neg")):
        an, mu, sg = S.nll(zt, zr, min_std=0.03, side=side, return_all=True)
        assert np.allclose(h(an) if tag == "pos" else g.sample(h(an)), g["nll_" + tag], rtol=1e-4, atol=1e-4), tag
    assert np.allclose(g.sample(h(mu)), g["nll_mu"], rtol=1e-6, atol=1e-6)
    assert np.allclose(g.sample(h(sg)), g["nll_sigma"], rtol=1e-5, atol=1e-6)
    assert np.allclose(g.sample(h(S.nll(zt, zr))), g["nll_eps"], rtol=1e-4, atol=1e-4)
    an_m = S.nll(zt, zr, min_std=0.03, side="+", mul_mask=g["in_valid"])
    assert np.allclose(h(an_m), g["nll_pos"] * g["in_valid"], rtol=1e-4, atol=1e-4)
    # masks per reference (image_ops.py:197-231) and the Otsu branch (reference code + the restated threshold_otsu)
    gm = list(g["gmask"])
    assert np.allclose(g.sample(h(S.group_mean(zr, gm))), g["group_mean_masked"], rtol=1e-6, atol=1e-6, equal_nan=True)
    assert np.allclose(g.sample(h(S.group_std(zr, gm))), g["group_std_masked"], rtol=1e-5, atol=1e-6, equal_nan=True)
    assert np.isnan(h(S.group_mean(zr, gm))[5:9]).all()
    an, mu, sg = S.nll(zt, zr, min_std=0.03, side="+", return_all=True, use_mask=True)
    assert np.allclose(g.sample(h(an)), g["nll_usemask"], rtol=1e-4, atol=1e-4)
    assert np.allclose(g.sample(h(mu)), g["nll_usemask_mu"], rtol=1e-6, atol=1e-6, equal_nan=True)
    assert np.allclose(g.sample(h(sg)), g["nll_usemask_sigma"], rtol=1e-5, atol=1e-6, equal_nan=True)
    with pytest.raises(ValueError):
        S.group_mean(zr, gm[:2])
    with pytest.raises(AssertionError):
        S.nll(zt, zr, side="x")
    with pytest.raises(Exception):
        S.nll(zt, [zr[0]] * 33)                                      # more references than the kernel's pointer table


@pytest.mark.parametrize("tag", ["p12", "p50", "podd", "nomask"])
def test_mean_std_grid_matches_reference_fixture(g, S, tag):
    if tag == "nomask":
        m, s = S.mean_std_grid(g["z_target"], [12, 12, 12])
    else:
        m, s = S.mean_std_grid(g["z_target"], g["msg_patch_" + tag].tolist(), mask=g["in_valid"])
    assert np.allclose(g.sample(h(m)), g["msg_mean_" + tag], rtol=1e-5, atol=2e-6)
    assert np.allclose(g.sample(h(s)), g["msg_std_" + tag], rtol=1e-5, atol=2e-6)
    with pytest.raises(NotImplementedError):
        S.mean_std_grid(g["z_target"], [12, 12, 12], order=3)


@pytest.mark.parametrize("tag", ["iso1", "iso07", "mixed", "thick"])
def test_median_3mm_bit_exact_with_reference_fixture(g, S, tag):
    vox = g["median_vox_" + tag].tolist()
    assert S.median_kernel_size(vox) == I.median_kernel(vox)
    assert np.array_equal(h(S.median_3mm(g["nll_pos"], vox)), g["median_" + tag])


def test_median_filter_edge_cases(S):
    rng = np.random.default_rng(3)
    for shape, ks in (((1, 1, 1), [3, 3, 3]), ((5, 3, 70), [1, 1, 1]), ((7, 9, 33), [9, 2, 5]), ((2, 70, 3), [3, 7, 1]),
                      # register-resident selection: odd and even (+inf padded) windows, every slice orientation
                      ((9, 21, 40), [4, 4, 4]), ((6, 37, 45), [1, 6, 6]), ((33, 5, 41), [6, 1, 6]), ((35, 38, 4), [6, 6, 1]),
                      ((30, 3, 33), [5, 1, 5]), ((17, 18, 5), [4, 4, 1]), ((3, 30, 31), [1, 5, 5]), ((20, 20, 20), [1, 3, 3])):
        x = rng.normal(size=shape).astype(np.float32)
        x[rng.random(shape) > 0.7] = 0.0                              # ties with the zero padding
        x[rng.random(shape) > 0.9] *= -1.0
        from scipy.ndimage import median_filter
        assert np.array_equal(h(S.median_filter(x, ks)), median_filter(x, size=ks, mode="constant", cval=0)), (shape, ks)
    with pytest.raises(Exception):
        S.median_filter(np.zeros((4, 4, 4), np.float32), [11, 3, 3])


def test_anomaly_pipeline_matches_reference_fixture(g, S):
    r = S.nll_anomaly_map(g["in_target"], list(g["in_refs"]), g["in_brain"], g["in_valid"], intensity_prior="+",
                          image_patch=g["pipe_patch"].tolist(), with_reference_scores=True)
    assert np.allclose(g.sample(h(r["normalized_input"])), g["pipe_x_prime"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(h(r["local_mean"])), g["pipe_local_mu"] * g.sample(g["in_valid"]), rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(h(r["mean"])), g["pipe_mean"], rtol=1e-5, atol=1e-5)
    assert np.allclose(g.sample(h(r["std"])), g["pipe_std"], rtol=1e-4, atol=1e-5)
    assert np.allclose(g.sample(h(r["anomaly"])), g["pipe_anomaly"], rtol=1e-4, atol=2e-3)
    assert np.allclose(g.sample(h(r["reference_anomalies"][0])), g["pipe_ref_anomaly0"], rtol=1e-4, atol=2e-3)
    # the lesion planted in the fixture's target is what the map finds
    assert np.unravel_index(np.argmax(h(r["anomaly"])), g["in_target"].shape)[0] in range(12, 16)


@pytest.mark.parametrize("tag", ["iso", "thick_z", "thick_x"])
def test_component_filtering_bit_exact_with_reference_fixture(g, S, tag):
    got = h(S.component_filtering(g["cf_in"], g["cf_vox_" + tag].tolist()))
    assert got.dtype == np.float32 and np.array_equal(got, g["cf_" + tag])


def test_component_filtering_edge_cases(g, S):
    assert np.array_equal(h(S.component_filtering(g["in_brain"], [1.0, 1.0, 1.0])), g["cf_brain"])
    assert h(S.component_filtering(np.zeros((6, 7, 5), np.float32), [1.0, 1.0, 1.0])).sum() == 0
    rng = np.random.default_rng(21)
    for shape, thr, vox in (((9, 31, 17), 0.35, [1.0, 1.0, 1.0]), ((40, 40, 40), 0.2, [1.0, 2.0, 1.5]), ((12, 50, 33), 0.3, [1.0, 3.5, 1.0]),
                            ((1, 20, 20), 0.2, [1.0, 1.0, 1.0]), ((64, 64, 48), 0.12, [0.8, 0.8, 0.8])):
        m = (rng.random(shape) > thr).astype(np.float32)              # many equal-size components: exercises the tie rule
        assert np.array_equal(h(S.component_filtering(m, vox)), I.component_filtering(m, vox)), (shape, vox)
    r = S.nll_anomaly_map(g["in_target"], list(g["in_refs"]), g["in_brain"], g["in_valid"], intensity_prior="+",
                          image_patch=g["pipe_patch"].tolist(), apply_component_filtering=True)
    assert np.allclose(g.sample(h(r["anomaly"])), g["pipe_anomaly_cf"], rtol=1e-4, atol=2e-3)
    with pytest.raises(NotImplementedError):
        S.component_filtering(g["in_brain"], [1.0, 1.0, 1.0], return_type="int")


def test_otsu_and_valid_score_mask(g, S):
    """threshold_otsu restates skimage's published algorithm (skimage is not vendored: unpinned); the device histogram is
    numpy.histogram bit for bit, so the threshold equals the numpy restatement on the same fp32 values exactly."""
    rng = np.random.default_rng(4)
    x = np.concatenate([rng.normal(-1, 0.3, 40000), rng.normal(2, 0.5, 25000)]).astype(np.float32).reshape(50, 50, 26)
    edges = np.linspace(float(x.min()), float(x.max()), 257)
    assert np.array_equal(S.histogram(x, edges), np.histogram(x.astype(np.float64), bins=edges)[0])
    assert S.minmax(x) == (float(x.min()), float(x.max()))
    assert S.threshold_otsu(x) == I.threshold_otsu(x) and -0.5 < S.threshold_otsu(x) < 1.5
    m = (rng.random(x.shape) > 0.4).astype(np.float32)
    assert np.array_equal(S.histogram(x, edges, mask=m), np.histogram(x[m > 0.5].astype(np.float64), bins=edges)[0])
    assert np.array_equal(S.histogram(x, edges, mask=m, fill_value=float(x.min())),
                          np.histogram(np.where(m > 0.5, x, x.min()).astype(np.float64), bins=edges)[0])
    assert S.otsu_thresholding(x, m) == I.threshold_otsu(x[m > 0.5])
    assert S.otsu_thresholding(x, np.zeros_like(m)) is None
    assert S.threshold_otsu(np.full((4, 4, 4), 3.5, np.float32)) == 3.5
    # values exactly on bin edges and the closed last bin
    e8 = np.linspace(0.0, 8.0, 9)
    v = np.array([0, 1, 1, 2, 7.9999995, 8, 8, 3.5, -1, 9], np.float32).reshape(1, 2, 5)
    assert np.array_equal(S.histogram(v, e8), np.histogram(v.astype(np.float64), bins=e8)[0])
    # lesion_analysis.py:142-148 on the fixture's raw target
    xp, valid = S.valid_score_mask(g["in_target"], g["in_brain"])
    xo, vo = I.valid_score_mask(g["in_target"], g["in_brain"])
    assert np.allclose(h(xp), xo, rtol=1e-5, atol=1e-5)
    xh, b = h(xp), g["in_brain"] >= 0.5
    thr = I.threshold_otsu(np.where(b, xh, xh.min()))                 # the restatement on the device's own fp32 z-scores
    assert np.array_equal(h(valid), (b * (xh > np.float32(thr))).astype(np.float32))
    assert (h(valid) != vo).mean() < 1e-2 and 0 < h(valid).sum() < g["in_brain"].sum()
    _, allv = S.valid_score_mask(g["in_target"], g["in_brain"], apply_otsu=False)
    assert np.array_equal(h(allv), (g["in_brain"] >= 0.5).astype(np.float32))


def test_batched_case_launches_equal_the_function_by_function_path(g, S):
    """dwmh_s1_zscore_batch / dwmh_s1_local_mean_align (whole case per launch) against z_score / mean_std_grid /
    align_local_mean_ called volume by volume."""
    brain, valid, patch = g["in_brain"], g["in_valid"], [14, 14, 14]
    vols = [torch.from_numpy(v.copy()).cuda() for v in [g["in_target"]] + list(g["in_refs"])]
    S.z_score_batch_(vols, brain, fill_outside=True)
    single = [S.z_score(v, brain, fill_outside=True) for v in [g["in_target"]] + list(g["in_refs"])]
    for a, b in zip(vols, single):
        assert np.allclose(h(a), h(b), rtol=0, atol=1e-6)               # fp64 atomics: summation order is free
    z0 = h(vols[0]).copy()
    mu_p = S.local_mean_align_(vols[0], vols[1:], patch, mask=valid)
    mu_ref, _ = S.mean_std_grid(single[0], patch, mask=valid)
    assert np.allclose(h(mu_p), h(mu_ref), rtol=0, atol=1e-6)          # fp64 atomics: summation order is free
    for a, b in zip(vols[1:], single[1:]):
        mu_i, _ = S.mean_std_grid(b, patch, mask=valid)
        S.align_local_mean_(b, mu_i, mu_ref)
        assert np.allclose(h(a), h(b), rtol=0, atol=2e-6)               # fused path skips the fp32 rounding of the two means
    assert np.array_equal(h(vols[0]), z0)                              # the target is read only
    # k = 0: local mean only; unmasked statistics; unaligned (odd-offset) views take the scalar kernels
    assert np.allclose(h(S.local_mean_align_(single[0], [], patch, mask=valid)), h(mu_ref), atol=1e-6)
    flat = torch.zeros(g["in_target"].size + 1, device="cuda")
    odd = flat[1:].view(g["in_target"].shape)
    odd.copy_(torch.from_numpy(g["in_target"]))
    S.z_score_batch_([odd], brain, fill_outside=True)
    assert np.allclose(h(odd), h(single[0]), rtol=0, atol=1e-6)
    with pytest.raises(ValueError):
        S.z_score_batch_([vols[0], vols[1][:-1]], brain)


def test_full_size_volume_against_oracle(S):
    """BASELINE.json's 182x218x182 shape, 1 mm isotropic: 50-voxel local-mean patch, 3x3x3 median."""
    import oracle as O
    shape = (182, 218, 182)
    tgt = O.synthetic_flair(shape, seed=0)[0]
    refs = [O.synthetic_flair(shape, seed=s)[0] for s in (1, 2, 3)]
    brain = (tgt != 0).astype(np.float32)
    valid = (brain * (np.random.default_rng(0).random(shape) > 0.05)).astype(np.float32)
    r = S.nll_anomaly_map(tgt, refs, brain, valid, physical_voxel_size=[1.0, 1.0, 1.0], intensity_prior="+")
    o = I.nll_anomaly_arrays(tgt, refs, brain, valid, S.image_patch_size([1.0, 1.0, 1.0]))
    assert np.allclose(h(r["normalized_input"]), o["x_prime"], rtol=1e-5, atol=1e-5)
    assert np.allclose(h(r["local_mean"]), o["local_mu"] * valid, rtol=1e-5, atol=1e-5)
    assert np.allclose(h(r["mean"]), o["mean"], rtol=1e-5, atol=1e-5)
    assert np.allclose(h(r["std"]), o["std"], rtol=1e-4, atol=1e-5)
    assert np.allclose(h(r["anomaly"]), o["anomaly"], rtol=1e-4, atol=2e-3)
    an32 = h(r["anomaly"])
    assert np.array_equal(h(S.median_3mm(an32, [1.0, 1.0, 1.0])), I.median_3mm(an32, [1.0, 1.0, 1.0]))
    # size-independent properties: z-scored statistics over the mask, constant fill outside, NLL floor
    z = h(r["normalized_input"])
    inside = z[brain > 0.5].astype(np.float64)
    assert abs(inside.mean()) < 1e-5 and abs(inside.std() - 1.0) < 1e-5
    assert np.unique(z[brain < 0.5]).size == 1 and z[brain < 0.5][0] == np.float32(inside.min())
    assert (h(r["std"]) >= np.float32(0.03)).all() and (an32[valid < 0.5] == 0).all()


@pytest.mark.parametrize("tag,prior", [("pos", "+"), ("none", None)])
def test_whole_nll_analysis_matches_the_reference_run_end_to_end(S, tag, prior):
    """tests/golden/nll_analysis_v1.npz holds what the reference's nll_analysis ITSELF returned and saved (run unmodified with
    its NIfTI I/O redirected to memory, apply_otsu=False); stage1.nll_analysis_arrays is the device path for the same arrays."""
    f = F.nll_analysis()
    an, valid, cx, cy, cr, thr, ex = S.nll_analysis_arrays(f["in_target"], list(f["in_refs"]), list(f["in_label1"]),
                                                           [t.astype(np.float32) for t in f["in_label2"]], f["voxel_size"].tolist(),
                                                           apply_otsu=False, intensity_prior=prior)
    assert np.array_equal(h(valid), f["valid_" + tag]) and np.array_equal(h(ex["rough_brain"]), f["rough_brain_" + tag])
    assert np.array_equal(h(ex["averaged_label"]), f["averaged_label_" + tag])
    assert np.allclose(f.sample(h(ex["normalized_input"])), f["normalized_input_" + tag], rtol=1e-5, atol=1e-5)
    assert np.allclose(f.sample(h(ex["local_mean"])), f["local_mean_" + tag], rtol=1e-5, atol=1e-5)
    assert np.allclose(f.sample(h(ex["mean"])), f["mean_value_" + tag], rtol=1e-5, atol=1e-5)
    assert np.allclose(f.sample(h(ex["std"]) * f["valid_" + tag]), f["std_value_" + tag], rtol=1e-4, atol=1e-5)
    assert np.allclose(h(an), f["anomaly_" + tag], rtol=1e-4, atol=2e-3)
    # histogram curves: a voxel whose score sits within fp32 rounding of a bin edge may change bins, which moves a
    # log10 count visibly only where counts are tiny -> all but a few of the 400 bins agree to 1e-2
    assert np.allclose(cx, f["curve_x_" + tag], rtol=1e-6)
    assert (np.abs(cy - f["curve_y_" + tag]) > 1e-2).sum() <= 4 and (np.abs(cr - f["curve_r_" + tag]) > 1e-2).sum() <= 4
    assert abs(thr - float(f["threshold_" + tag])) <= 1.01 * (cx[1] - cx[0])
    a = h(an)
    assert a[20:23, 12:15, 6:9].max() > thr and a[14:18, 22:27, 20:24].max() > thr          # both planted lesions are found
