"""Models with M input modalities and C classes (nnU-Net v1 3d_fullres beyond DeepWMH's M = 1, C = 2).

Random-init oracle networks for (M, C) in {(2, 3) WMH-challenge layout (T1 + FLAIR; background, WMH, other pathology),
(4, 4), (1, 3), (3, 2)}, on a 3^3 plan (first conv on tcgen05) and an anisotropic plan (1x3x3 first conv, CUDA cores):
  * dwmh_forward_patches against the fp32 oracle, and against the CUDA-core kernels (dwmh_set_force_generic);
  * every layer and the head against float64 references fed the device's own inputs (tests/test_gpu_layer_fp64.py's
    rounding model) for every class count 3..8, in fp16 and bf16, with base 32 (the head's two-voxel branch) and 64 (its
    one-voxel branch), plus a negative check: the reference without one modality's taps must fail the tolerance;
  * tiled predict_3D with 8x mirroring on a volume larger than the patch, against the oracle's predict_3D;
  * volumes smaller than the patch: numpy and CUDA input padded alike, against a float64 aggregation of the padded volume;
  * the host-buffer call against normalize_ + predict_3D, bit for bit (padding, re-pitched modalities, crop mask);
  * the resident ensemble, the tile-sharded call in one process and the weight map at C = 3;
  * determinism: two calls are bit-identical, split tile ranges add up to the full run;
  * argmax and both paths of finalize (128-bit and scalar) pick the lower class on planted ties, two classes included;
  * accumulate_tiles / finalize refuse tensors the kernels cannot take;
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
import test_gpu_tiling_fp64 as TT
from test_gpu_layer_fp64 import U, _first_conv, _instnorm_lrelu, check_reports, conv_report, layer_fp64_reports, rounded_copy

pytestmark = pytest.mark.gpu

MC = [(2, 3), (4, 4), (1, 3), (3, 2)]
SOFTMAX_TOL, AGREE_MIN = 2e-2, 0.999


def _plans(kind, M, C, base=32):
    if kind == "cube":
        p = small_plans(base=base)
    else:
        p = small_plans(patch=(16, 64, 48), pools=((1, 2, 2), (2, 2, 2), (2, 2, 2)), kernels=[[1, 3, 3], [3, 3, 3], [3, 3, 3], [3, 3, 3]],
                        base=base)
    p["num_modalities"], p["num_classes"] = M, C - 1
    p["normalization_schemes"] = {m: "nonCT" for m in range(M)}
    p["use_mask_for_norm"] = {m: True for m in range(M)}
    return p


def _pair(kind, M, C, max_batch=8, seed=0, base=32, act="fp16"):
    import deepwmh_b200
    plans = _plans(kind, M, C, base)
    net = O.build_benchmark_network(seed, plans)
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, act_dtype=act, max_batch=max_batch)
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


# (kind, M, C, base_num_features, activation type).  Every head class count 3..8; (4, 8) is the head's largest shared
# memory and register footprint; bf16 with several modalities takes the MULTI first conv's bf16 hi / lo split on the cube
# plan and conv_first_mm_kernel's bf16 instantiation on the anisotropic one; base 64 gives the head a 64-channel input,
# its one-voxel (scalar) branch.
LAYER_CASES = [
    ("cube", 2, 3, 32, "fp16"), ("aniso", 2, 3, 32, "fp16"), ("cube", 4, 4, 32, "fp16"), ("aniso", 4, 4, 32, "fp16"),
    ("cube", 3, 5, 32, "fp16"), ("aniso", 2, 6, 32, "fp16"), ("cube", 1, 7, 32, "fp16"), ("cube", 4, 8, 32, "fp16"),
    ("cube", 2, 3, 32, "bf16"), ("aniso", 4, 4, 32, "bf16"), ("cube", 3, 8, 32, "bf16"),
    ("cube", 1, 3, 64, "fp16"), ("cube", 1, 8, 64, "fp16"),
]


def _layer_case_id(case):
    kind, M, C, base, act = case
    # the fp16, base-32 cases keep the ids of the (M, C) x kind grid they came from
    return "-".join([str(M), str(C), kind] + (["base%d" % base] if base != 32 else []) + ([act] if act != "fp16" else []))


@pytest.mark.parametrize("kind,M,C,base,act", LAYER_CASES, ids=[_layer_case_id(c) for c in LAYER_CASES])
def test_layers_match_fp64_and_see_a_dropped_modality(kind, M, C, base, act):
    plans, net, tr = _pair(kind, M, C, base=base, act=act)
    dev = tr.network
    x = _patches(2, M, dev.patch_size, seed=7 + M).cuda()
    reports, head = layer_fp64_reports(net, dev, x, act)
    check_reports(_layer_case_id((kind, M, C, base, act)), reports, head)
    # negative check: the first conv's reference without the taps of one modality must exceed the tolerance
    ref_net = rounded_copy(net, act, torch.float64, x.device)
    m0 = _first_conv(ref_net)
    xd = x.to(torch.float64)
    got = dev.layer_output(0, 2).to(torch.float64)
    for drop in range(M if M > 1 else 0):
        xm = xd.clone()
        xm[:, drop] = 0.0
        with torch.no_grad():
            y = m0.conv(xm)
            err, _ = conv_report(m0, xm, y, _instnorm_lrelu(y, m0), got, U[act], U[act])
        print("%s M=%d %s: without modality %d  max err/tol %.1f" % (kind, M, act, drop, err))
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


# the anisotropic plan's first conv runs on CUDA cores: conv_first_mm_kernel (M > 1), conv_first_kernel (M = 1)
@pytest.mark.parametrize("kind,M,C", [("cube", 2, 3), ("cube", 4, 4), ("aniso", 2, 3), ("aniso", 1, 3)],
                         ids=["2-3", "4-4", "aniso-2-3", "aniso-1-3"])
def test_bit_identical_repeat_and_split_tile_ranges(kind, M, C):
    plans, net, tr = _pair(kind, M, C)
    dev = tr.network
    rng = np.random.default_rng(5)
    shp = (48, 40, 40) if kind == "cube" else (24, 70, 60)
    vol = torch.from_numpy(rng.normal(size=(M,) + shp).astype(np.float32)).cuda()

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


# (20, 16, 13) takes finalize's 128-bit path, the odd voxel count of (19, 17, 13) its scalar one
@pytest.mark.parametrize("C,shp", [(C, (20, 16, 13)) for C in (3, 5, 8, 2)] + [(C, (19, 17, 13)) for C in (2, 3, 8)],
                         ids=["3", "5", "8", "2", "2-odd", "3-odd", "8-odd"])
def test_argmax_and_finalize_break_ties_to_the_lower_class(C, shp):
    import deepwmh_b200
    plans, net, tr = _pair("cube", 1, C)
    dev = tr.network
    rng = np.random.default_rng(C)
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


# volumes smaller than the 32^3 patch along one, two and three axes
@pytest.mark.parametrize("shape", [(24, 40, 36), (20, 28, 40), (25, 30, 31)])
@pytest.mark.parametrize("M,C", [(2, 3), (4, 4)])
def test_padded_volume_from_numpy_and_cuda_input_matches_fp64_aggregation(M, C, shape):
    """predict_3D pads numpy input with pad_nd_image and CUDA input with F.pad: both must give the same bits, and match
    the float64 reconstruction of the zero-padded volume (d // 2 below, d // 2 + d % 2 above) cropped back."""
    plans, net, tr = _pair("cube", M, C)
    dev = tr.network
    x = TT._volume_np(shape, M, seed=M + C)
    seg_n, p_n = dev.predict_3D(x, True, use_sliding_window=True, step_size=0.5, use_gaussian=True)
    seg_c, p_c = dev.predict_3D(torch.from_numpy(x).cuda(), True, use_sliding_window=True, step_size=0.5, use_gaussian=True)
    assert p_n.shape == (C,) + shape and seg_n.shape == shape
    assert np.array_equal(p_n, p_c) and np.array_equal(seg_n, seg_c)
    pads = [(max(p - s, 0) // 2, max(p - s, 0) // 2 + max(p - s, 0) % 2) for p, s in zip(dev.patch_size, shape)]
    vol = torch.from_numpy(np.pad(x, [(0, 0)] + pads)).cuda()
    rec = TT.Reconstruction(dev, vol, 0.5, True, (0, 1, 2), True, 8)
    p_ref, _ = rec.aggregate()
    p_ref = p_ref[(slice(None),) + tuple(slice(b, b + s) for (b, _), s in zip(pads, shape))]
    err = (torch.from_numpy(p_n).cuda().double() - p_ref).abs().max().item()
    seg_bad = TT.label_mismatches(torch.from_numpy(seg_n).cuda(), p_ref)
    print("padded %s M=%d C=%d: tiles %d  softmax max|d| %.2e (%.3f of tol)  seg mismatches %d"
          % ("x".join(map(str, shape)), M, C, len(rec.origins), err, err / TT.SOFTMAX_TOL, seg_bad))
    assert err <= TT.SOFTMAX_TOL and seg_bad == 0
    dev.close()


# (M, C, shape, crop mask): X Y Z % 4 == 0 and != 0 (the host call re-pitches the modalities to 16-byte aligned
# channels), unpadded and smaller than the patch, z-score over vol != 0 and over a crop mask shared by all modalities
HOST_CASES = [(2, 3, (40, 36, 34), False), (2, 3, (35, 33, 37), False), (2, 3, (24, 40, 36), False),
              (2, 3, (25, 33, 35), False), (2, 3, (35, 33, 37), True), (2, 3, (24, 40, 36), True), (4, 4, (25, 33, 35), True)]


@pytest.mark.parametrize("M,C,shape,masked", HOST_CASES)
def test_host_buffer_call_equals_device_call_with_several_modalities(M, C, shape, masked):
    """predict_raw_volume_host (z-score per modality, padding and the per-class copy back inside the library) against
    normalize_ of each modality followed by predict_3D on the device tensor: bit-identical."""
    plans, net, tr = _pair("cube", M, C)
    dev = tr.network
    raw = np.stack([O.synthetic_flair(shape, seed=20 + m)[0] * (1.0 + m) for m in range(M)]).astype(np.float32)
    mask = None
    if masked:
        mask = np.full(shape, -1, np.int8)
        mask[2:-2, 3:-3, 1:-1] = 0
    seg_h, p_h = tr.predict_raw_volume_host(raw, seg_mask=mask)
    vols = []
    for m in range(M):
        v = torch.from_numpy(raw[m].copy()).cuda()          # its own tensor: dwmh_zscore needs 16-byte aligned channels
        dev.normalize_(v, torch.from_numpy(mask).cuda() if masked else None, 1 if masked else 2)
        vols.append(v)
    seg_d, p_d = dev.predict_3D(torch.stack(vols), True, use_sliding_window=True, step_size=0.5, use_gaussian=True)
    print("host call M=%d C=%d %s%s: max |p_host - p_device| %.1e" % (M, C, "x".join(map(str, shape)), " masked" if masked else "",
                                                                     np.abs(p_h - p_d).max()))
    assert p_h.shape == (C,) + shape
    assert np.array_equal(p_h, p_d) and np.array_equal(seg_h, seg_d.astype(np.uint8))
    dev.close()


def test_ensemble_mean_of_three_resident_models():
    """predict_volume_ensemble (three (2, 3) models sharing one workspace): the mean is the fp32 running mean
    mean += softmax_k / 3 of separate runs (the library fuses multiply and add, the reference rounds twice: 1e-6), and the
    label is numpy.argmax of the mean."""
    from deepwmh_b200 import parallel
    M, C = 2, 3
    plans = _plans("cube", M, C)
    trs = parallel.make_ensemble(plans, [O.build_benchmark_network(s, plans).state_dict() for s in range(3)], max_batch=8)
    vol = torch.from_numpy(TT._volume_np((40, 50, 45), M)).cuda()
    seg, mean = parallel.predict_volume_ensemble(trs, vol)
    ref = torch.zeros_like(mean)
    for tr in trs:
        _, p = tr.network.predict_3D(vol, True, use_sliding_window=True, step_size=0.5, use_gaussian=True,
                                     return_device_tensors=True)
        ref = ref + (1.0 / 3) * p
    err = (mean - ref).abs().max().item()
    print("ensemble of 3 M=%d C=%d: max |mean - running mean of runs| %.1e" % (M, C, err))
    assert mean.shape == (C, 40, 50, 45) and err <= 1e-6
    assert np.array_equal(seg.cpu().numpy(), mean.cpu().numpy().argmax(0))
    assert TT.label_mismatches(seg, ref.double()) == 0
    for tr in reversed(trs):
        tr.network.close()


def test_tile_sharded_call_equals_predict_3d_and_weight_map_equals_the_tiles_sum():
    """One process (world size 1): predict_volume_tile_sharded replaces the accumulated weights with dwmh_weight_map,
    which must be the same bits for a three-class model."""
    from deepwmh_b200 import parallel
    plans, net, tr = _pair("cube", 2, 3)
    dev = tr.network
    shp = (40, 50, 45)
    vol = torch.from_numpy(TT._volume_np(shp, 2)).cuda()
    seg_s, p_s = parallel.predict_volume_tile_sharded(tr, vol)
    seg_d, p_d = dev.predict_3D(vol, True, use_sliding_window=True, step_size=0.5, use_gaussian=True, return_device_tensors=True)
    assert p_s.shape == (3,) + shp
    assert torch.equal(p_s, p_d) and torch.equal(seg_s, seg_d)
    agg = torch.zeros((3,) + shp, device="cuda")
    wgt = torch.zeros(shp, device="cuda")
    dev.accumulate_tiles(vol, agg, wgt, 0.5, True, (0, 1, 2), True)
    assert torch.equal(dev.weight_map(shp, 0.5, True), wgt)
    dev.close()


def test_accumulate_tiles_and_finalize_reject_tensors_the_kernels_cannot_take():
    """The kernels take raw pointers: host tensors, other dtypes, strided views and wrong shapes are refused before any
    launch (the buffers stay untouched)."""
    plans, net, tr = _pair("cube", 2, 3)
    dev = tr.network
    shp = (40, 36, 34)
    vol = torch.ones((2,) + shp, device="cuda")
    agg = torch.zeros((3,) + shp, device="cuda")
    wgt = torch.zeros(shp, device="cuda")
    strided = lambda t: torch.zeros(tuple(t.shape) + (2,), device="cuda")[..., 0]
    bad = {
        "vol on the host": dict(vol=vol.cpu()), "vol float64": dict(vol=vol.double()), "vol strided": dict(vol=strided(vol)),
        "vol one modality": dict(vol=vol[:1]), "vol [X, Y, Z]": dict(vol=vol[0]),
        "vol of another volume": dict(vol=vol[:, :, :, :-1].contiguous()),
        "agg on the host": dict(agg=agg.cpu()), "agg float16": dict(agg=agg.half()), "agg strided": dict(agg=strided(agg)),
        "agg two classes": dict(agg=agg[:2]), "agg [X, Y, Z]": dict(agg=agg[0]),
        "wgt on the host": dict(wgt=wgt.cpu()), "wgt float64": dict(wgt=wgt.double()), "wgt strided": dict(wgt=strided(wgt)),
        "wgt short": dict(wgt=wgt[:-1]), "wgt [1, X, Y, Z]": dict(wgt=wgt[None]),
    }
    for what, repl in bad.items():
        a = {**dict(vol=vol, agg=agg, wgt=wgt), **repl}
        with pytest.raises(ValueError):
            dev.accumulate_tiles(a["vol"], a["agg"], a["wgt"], 0.5, True, (0, 1, 2), True)
        if "vol" not in repl:
            with pytest.raises(ValueError):
                dev.finalize(a["agg"], a["wgt"])
        print("rejected:", what)
    torch.cuda.synchronize()
    assert not agg.any() and not wgt.any()
    dev.accumulate_tiles(vol, agg, wgt, 0.5, False, (), True, 0, 1)     # the intact buffers are still accepted
    seg, p = dev.finalize(agg, wgt)
    assert seg.shape == shp and p.data_ptr() == agg.data_ptr()
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
