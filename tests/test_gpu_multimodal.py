"""Models with M input modalities and C classes (nnU-Net v1 3d_fullres beyond DeepWMH's M = 1, C = 2).

Random-init oracle networks for (M, C) in {(2, 3) WMH-challenge layout (T1 + FLAIR; background, WMH, other pathology),
(4, 4), (1, 3), (3, 2)}, on a 3^3 plan (first conv on tcgen05) and an anisotropic plan (1x3x3 first conv, CUDA cores):
  * dwmh_forward_patches against the fp32 oracle, and against the CUDA-core kernels (dwmh_set_force_generic);
  * every layer and the head against float64 references fed the device's own inputs (tests/test_gpu_layer_fp64.py's
    rounding model), plus a negative check: the reference without one modality's taps must fail the tolerance;
  * tiled predict_3D with 8x mirroring on a volume larger than the patch, against the oracle's predict_3D;
  * determinism: two calls are bit-identical, split tile ranges add up to the full run;
  * argmax over C classes on planted ties picks the lower class;
  * nnUNet_predict end to end on a 2-modality, 3-class model directory against the oracle pipeline.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle as O
import oracle.resample_oracle as R
from conftest import small_plans
from test_gpu_layer_fp64 import U, _first_conv, _instnorm_lrelu, check_reports, conv_report, layer_fp64_reports, rounded_copy

pytestmark = pytest.mark.gpu

MC = [(2, 3), (4, 4), (1, 3), (3, 2)]
SOFTMAX_TOL, AGREE_MIN = 2e-2, 0.999


def _plans(kind, M, C):
    if kind == "cube":
        p = small_plans()
    else:
        p = small_plans(patch=(16, 64, 48), pools=((1, 2, 2), (2, 2, 2), (2, 2, 2)), kernels=[[1, 3, 3], [3, 3, 3], [3, 3, 3], [3, 3, 3]])
    p["num_modalities"], p["num_classes"] = M, C - 1
    p["normalization_schemes"] = {m: "nonCT" for m in range(M)}
    p["use_mask_for_norm"] = {m: True for m in range(M)}
    return p


def _pair(kind, M, C, max_batch=8, seed=0):
    import deepwmh_b200
    plans = _plans(kind, M, C)
    net = O.build_benchmark_network(seed, plans)
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=max_batch)
    tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
    return plans, net, tr


def _patches(n, M, patch, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((n, M) + tuple(patch), generator=g)
    x[:, :, :2] = 0.0                                            # some zero background, as z-scored volumes have
    return x


@pytest.mark.parametrize("kind", ["cube", "aniso"])
@pytest.mark.parametrize("M,C", MC)
def test_forward_patches_match_oracle_and_cuda_core(kind, M, C):
    plans, net, tr = _pair(kind, M, C)
    dev = tr.network
    assert dev.num_classes == C and dev.input_channels == M
    if kind == "cube":
        assert dev.layer_kernel_kind(0) == 1, "3x3x3 first conv must run on tcgen05"
    x = _patches(4, M, dev.patch_size, seed=10 * M + C)
    with torch.no_grad():
        ref = torch.softmax(net.float()(x), 1).numpy()
    got = dev.forward_patches(x.cuda()).cpu().numpy()
    assert got.shape == (4, C) + tuple(dev.patch_size)
    assert np.allclose(got.sum(1), 1.0, atol=1e-5)
    err = np.abs(got - ref).max()
    agree = np.mean(got.argmax(1) == ref.argmax(1))
    print("%s M=%d C=%d  max |p - p_oracle| %.2e  argmax agreement %.5f" % (kind, M, C, err, agree))
    assert err < SOFTMAX_TOL and agree >= 0.995
    dev.set_force_generic(True)
    try:
        gen = dev.forward_patches(x.cuda()).cpu().numpy()
    finally:
        dev.set_force_generic(False)
    assert np.abs(gen - got).max() < SOFTMAX_TOL / 2, np.abs(gen - got).max()
    dev.close()


@pytest.mark.parametrize("kind", ["cube", "aniso"])
@pytest.mark.parametrize("M,C", [(2, 3), (4, 4)])
def test_layers_match_fp64_and_see_a_dropped_modality(kind, M, C):
    plans, net, tr = _pair(kind, M, C)
    dev = tr.network
    x = _patches(2, M, dev.patch_size, seed=7 + M).cuda()
    reports, head = layer_fp64_reports(net, dev, x)
    check_reports("%s M=%d C=%d" % (kind, M, C), reports, head)
    # negative check: the first conv's reference without the taps of one modality must exceed the tolerance
    ref_net = rounded_copy(net, "fp16", torch.float64, x.device)
    m0 = _first_conv(ref_net)
    xd = x.to(torch.float64)
    got = dev.layer_output(0, 2).to(torch.float64)
    for drop in range(M):
        xm = xd.clone()
        xm[:, drop] = 0.0
        with torch.no_grad():
            y = m0.conv(xm)
            err, _ = conv_report(m0, xm, y, _instnorm_lrelu(y, m0), got, U["fp16"], U["fp16"])
        print("%s M=%d: without modality %d  max err/tol %.1f" % (kind, M, drop, err))
        assert err > 1.0, (drop, err)
    dev.close()


@pytest.mark.parametrize("M,C", MC)
def test_tiled_predict_3d_with_tta_matches_oracle(M, C):
    plans, net, tr = _pair("cube", M, C, max_batch=16)
    rng = np.random.default_rng(M * 10 + C)
    x = rng.normal(size=(M, 50, 45, 41)).astype(np.float32)
    x[:, :3] = 0.0
    seg, p = tr.network.predict_3D(x, True, use_sliding_window=True, step_size=0.5, use_gaussian=True)
    seg_r, p_r = O.OracleTrainer(plans, net.float()).predict_preprocessed_data_return_seg_and_softmax(x, do_mirroring=True)
    assert p.shape == (C, 50, 45, 41) and seg.shape == (50, 45, 41)
    err, agree = np.abs(p - p_r).max(), np.mean(seg == seg_r)
    print("M=%d C=%d  predict_3D max |p - p_oracle| %.2e  argmax agreement %.5f" % (M, C, err, agree))
    assert err <= SOFTMAX_TOL and agree >= AGREE_MIN
    assert seg.max() < C and np.array_equal(seg, p.argmax(0))
    tr.network.close()


@pytest.mark.parametrize("M,C", [(2, 3), (4, 4)])
def test_bit_identical_repeat_and_split_tile_ranges(M, C):
    plans, net, tr = _pair("cube", M, C)
    dev = tr.network
    rng = np.random.default_rng(5)
    vol = torch.from_numpy(rng.normal(size=(M, 48, 40, 40)).astype(np.float32)).cuda()
    shp = (48, 40, 40)

    def run(ranges):
        agg = torch.zeros((C,) + shp, device="cuda")
        wgt = torch.zeros(shp, device="cuda")
        for b, e in ranges:
            dev.accumulate_tiles(vol, agg, wgt, 0.5, True, (0, 1, 2), True, b, e)
        return agg, wgt

    n = dev.num_tiles(shp, 0.5)
    a1, w1 = run([(0, -1)])
    a2, w2 = run([(0, -1)])
    assert torch.equal(a1, a2) and torch.equal(w1, w2)
    a3, w3 = run([(0, n // 3), (n // 3, n)])
    assert torch.equal(a1, a3) and torch.equal(w1, w3)
    dev.close()


@pytest.mark.parametrize("C", [3, 5, 8])
def test_argmax_and_finalize_break_ties_to_the_lower_class(C):
    import deepwmh_b200
    plans, net, tr = _pair("cube", 1, C)
    dev = tr.network
    rng = np.random.default_rng(C)
    shp = (20, 16, 13)
    p = rng.random((C,) + shp).astype(np.float32)
    # plant ties: a random pair of classes shares the maximum at a quarter of the voxels, all classes tie at a few
    tie = rng.random(shp) < 0.25
    a, b = rng.integers(0, C, size=shp), rng.integers(0, C, size=shp)
    mx = p.max(0) + 1.0
    for c in range(C):
        p[c][tie & ((a == c) | (b == c))] = mx[tie & ((a == c) | (b == c))]
    p[:, :2, :2, :2] = 0.5
    ref = p.argmax(0)                                              # numpy: first maximum
    pd = torch.from_numpy(p).cuda()
    assert np.array_equal(dev.argmax(pd).cpu().numpy(), ref)
    wgt = torch.from_numpy(rng.random(shp).astype(np.float32) + 0.5).cuda()
    agg = (pd * wgt).contiguous()
    seg, probs = dev.finalize(agg.clone(), wgt)
    pr = (agg / wgt).cpu().numpy()
    assert np.array_equal(probs.cpu().numpy(), pr)
    assert np.array_equal(seg.cpu().numpy(), pr.argmax(0))
    dev.close()


def test_nnunet_predict_two_modalities_three_classes_end_to_end(tmp_path, monkeypatch):
    """T1 + FLAIR, three classes, through `nnUNet_predict` against crop -> resample -> z-score -> oracle predict_3D ->
    resample back -> argmax -> paste back."""
    from deepwmh_b200 import nifti, nnunet_predict as NP, preprocess
    from test_resample import _make_model_dir
    M, C = 2, 3
    plans = _plans("cube", M, C)
    plans["plans_per_stage"][0]["current_spacing"] = np.array([1.2, 1.0, 1.0])
    net = O.build_benchmark_network(3, plans)
    root = str(tmp_path / "model")
    _make_model_dir(root, plans, net)
    vols = []
    for m in range(M):
        v = np.zeros((30, 44, 40), np.float32)
        v[2:28, 3:41, 4:37] = O.synthetic_flair((26, 38, 33), seed=40 + m)[0] * (1.0 + 0.5 * m)
        vols.append(v)
    vols[1][10:12, 20:22, 20:22] = 0.0                           # a hole in one modality only: the union mask keeps it
    indir = tmp_path / "in"; indir.mkdir()
    hdr = nifti.default_header((40, 44, 30), spacing=(1.0, 1.0, 1.1))
    for m in range(M):
        nifti.write_nifti(str(indir / ("caseB_%04d.nii.gz" % m)), np.transpose(vols[m], (2, 1, 0)), hdr)
    monkeypatch.setenv("RESULTS_FOLDER", root)
    out = str(tmp_path / "out")
    argv = ["-i", str(indir), "-o", out, "-t", "Task002_FinalModel", "-f", "all", "-chk", "model_best", "--save_softmax"]
    assert NP.main(argv) == 0
    seg_xyz, _ = nifti.read_nifti(os.path.join(out, "caseB.nii.gz"))
    seg = np.transpose(seg_xyz, (2, 1, 0))
    # oracle pipeline
    data = np.stack(vols)
    spacing = np.array([1.1, 1.0, 1.0])
    cropped, cseg, bbox = preprocess.crop_to_nonzero(data)
    target = np.array(plans["plans_per_stage"][0]["current_spacing"])
    d, _ = R.resample_and_normalize(cropped, cseg, spacing, target, True)
    _, sm = O.OracleTrainer(plans, net.float()).predict_preprocessed_data_return_seg_and_softmax(d.astype(np.float32), do_mirroring=True)
    sm = R.resample_softmax_back(sm, cropped.shape[1:], spacing, target)
    ref = preprocess.paste_back(sm.argmax(0).astype(np.uint8), data.shape[1:], bbox)
    agree = np.mean(seg == ref)
    print("nnUNet_predict M=2 C=3: label agreement %.5f, labels %s" % (agree, np.unique(seg)))
    assert seg.max() <= C - 1 and agree > 0.997
    assert os.path.isfile(os.path.join(out, "caseB_0.nii.gz"))
