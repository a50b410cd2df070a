"""CPU: the N4 restatement (oracle/n4_oracle.py) holds the properties the algorithm guarantees -- exact lattice refinement,
an identity sharpening for a vanishing FWHM, scale equivariance, pass-through of voxels <= 0 -- and recovers a known
bias field on a phantom; the --device-bfc command-line option is exclusive with --skip-bfc and has no CPU fallback."""
import os
import pickle

import numpy as np
import pytest
import torch

import oracle as O
from conftest import small_plans
from deepwmh_b200 import cli, nifti
from oracle import n4_oracle as N


def test_knot_insertion_reproduces_the_coarse_field():
    rng = np.random.default_rng(0)
    for mesh, n in ((1, 40), (2, 91), (4, 218), (8, 23)):
        phi = rng.normal(size=(mesh + 3,) * 3)
        pts = [np.sort(rng.integers(0, n, 17)) for _ in range(3)]
        coarse = N.evaluate(phi, *[N.basis_matrix(p, n, mesh) for p in pts])
        fine = N.evaluate(N.refine(phi), *[N.basis_matrix(p, n, 2 * mesh) for p in pts])
        assert np.abs(coarse - fine).max() <= 1e-12, mesh


def test_basis_is_a_partition_of_unity_with_four_taps():
    for mesh, n in ((1, 5), (4, 91), (8, 182)):
        w = N.basis_matrix(np.arange(n), n, mesh)
        assert w.shape == (n, mesh + 3)
        assert np.allclose(w.sum(1), 1.0, atol=1e-15, rtol=0) and ((w > 0).sum(1) <= 4).all()


def test_sharpening_with_a_vanishing_fwhm_is_the_identity_on_bin_centres():
    rng = np.random.default_rng(1)
    lo, hi = 2.0, 7.0
    slope = (hi - lo) / (N.BINS - 1)
    hist = rng.uniform(1.0, 50.0, N.BINS)
    e = N.sharpen_table(hist, lo, slope, fwhm=1e-3 * slope)
    centres = lo + np.arange(N.BINS) * slope
    assert np.abs(e - centres).max() <= 1e-6 * (hi - lo)


@pytest.mark.parametrize("alpha", [0.5, 7.0])
def test_scale_equivariance(alpha):
    """log(alpha I) shifts U by log(alpha): the histogram range moves with it and the residual does not change."""
    img, _, _ = N.phantom((40, 36, 32), seed=2)
    sched = (6, 6)
    base, f0 = N.n4(img, 2, sched, return_log_field=True)
    scaled, f1 = N.n4(img.astype(np.float64) * alpha, 2, sched, return_log_field=True)
    v = img > 0
    assert np.abs(scaled[v] - alpha * base[v]).max() <= 1e-10 * np.abs(alpha * base[v]).max()
    assert np.abs(f1 - f0).max() <= 1e-10


def test_voxels_at_or_below_zero_pass_through():
    img, _, _ = N.phantom((36, 32, 30), seed=3)
    img = img.astype(np.float64)
    img[:4, :4, :4] = -5.0
    out, field = N.n4(img, 2, (5, 5), return_log_field=True)
    assert np.array_equal(out[img == 0], img[img == 0])
    neg = img < 0
    assert np.allclose(out[neg], img[neg] / np.exp(field[neg]), rtol=1e-15, atol=0)
    # voxels <= 0 do not influence the fit: a different negative value leaves the field unchanged
    img2 = img.copy()
    img2[:4, :4, :4] = -1e6
    _, field2 = N.n4(img2, 2, (5, 5), return_log_field=True)
    assert np.array_equal(field, field2)


def test_phantom_recovery():
    """64^3 phantom, shrink 2, 20 iterations on each of three levels.  Measured with the oracle: worst within-class
    coefficient of variation 0.0700 -> 0.0302 (ratio 0.43; the multiplicative noise alone is 0.03), Pearson correlation of
    the recovered log field with the true one 0.9934."""
    img, f, labels = N.phantom((64, 64, 64), seed=1)
    out, field = N.n4(img, 2, (20, 20, 20), return_log_field=True)
    v = labels > 0

    def worst_cv(a):
        return max(np.std(a[labels == k]) / np.mean(a[labels == k]) for k in (1, 2, 3))
    assert worst_cv(out) < 0.5 * worst_cv(img)
    assert np.corrcoef(field[v], f[v])[0, 1] >= 0.95


def test_shrink_keeps_the_voxel_nearest_each_block_centre():
    assert N.shrink_indices(7, 2).tolist() == [1, 3, 5]
    assert N.shrink_indices(10, 3).tolist() == [1, 4, 7]
    assert N.shrink_indices(5, 1).tolist() == [0, 1, 2, 3, 4]
    with pytest.raises(ValueError):
        N.n4(np.ones((3, 8, 8), np.float32), 2, (1,))


def _model_dir(root):
    plans = small_plans()
    net = O.build_benchmark_network(0, plans)
    tdir = os.path.join(root, "nnUNet", "3d_fullres", "Task002_FinalModel", "nnUNetTrainerV2__nnUNetPlansv2.1")
    os.makedirs(os.path.join(tdir, "all"))
    pickle.dump(plans, open(os.path.join(tdir, "plans.pkl"), "wb"))
    torch.save({"epoch": 1, "state_dict": net.state_dict()}, os.path.join(tdir, "all", "model_best.model"))
    return plans, net


def test_cli_device_bfc_is_exclusive_with_skip_bfc(tmp_path):
    root = str(tmp_path / "model")
    _model_dir(root)
    img = str(tmp_path / "a.nii.gz")
    nifti.write_nifti(img, np.ones((8, 8, 8), np.float32), nifti.default_header((8, 8, 8)))
    with pytest.raises(SystemExit) as e:
        cli.main(["-i", img, "-n", "a", "-m", root, "-o", str(tmp_path / "o"), "--skip-bfc", "--device-bfc"])
    assert e.value.code == 2


def test_cli_device_bfc_without_a_gpu_fails_loudly(tmp_path, monkeypatch):
    root = str(tmp_path / "model")
    _model_dir(root)
    img = str(tmp_path / "a.nii.gz")
    nifti.write_nifti(img, np.ones((8, 8, 8), np.float32), nifti.default_header((8, 8, 8)))
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(RuntimeError, match="GPU only"):
        cli.main(["-i", img, "-n", "a", "-m", root, "-o", str(tmp_path / "o"), "--device-bfc"])
    assert not os.path.exists(str(tmp_path / "o" / "001_Preprocessed_Images" / "a_0000.nii.gz"))
