"""Region-based models (sigmoid outputs, regions_class_order; nnUNetTrainerV2BraTSRegions, DESIGN §12) on the B200.

BraTS-like layouts: four modalities and three region outputs on the small cube plan (tcgen05 first conv), the anisotropic
plan (CUDA-core first conv) and the 128^3 benchmark plan; other output counts on the cube plan for the head.
  * dwmh_forward_patches against the fp32 oracle (sigmoid per output) and against the CUDA-core kernels;
  * the sigmoid head against a float64 reference fed the device's own last-layer output, with negative checks: a swapped
    coefficient chunk and a softmax in place of the sigmoid must exceed the tolerance;
  * the overlap-add bit for bit against a float32 restatement of the reference's `*=` / `+=` fed the device's own forwards;
  * dwmh_region_labels bit for bit against numpy on device probabilities with planted 0.5 / +-1 ulp / NaN values;
  * tiled predict_3D with 8x mirroring against the oracle's region predictor; bit-identical repeats and split tile ranges;
  * nnUNet_predict -tr nnUNetTrainerV2BraTSRegions end to end with a resample and a postprocessing.json.
"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle as O
import oracle.resample_oracle as R
import postprocessing_oracle as PO
import regions_oracle as RO
import test_gpu_tiling_fp64 as TT
from test_gpu_layer_fp64 import _sub, swap_last_class_chunks
from test_gpu_multimodal import _patches, _plans

pytestmark = pytest.mark.gpu

PROB_TOL, AGREE_MIN = 2e-2, 0.995
ORDER = (1, 2, 3)
SENS_MIN = 4.0


def _brats_plans(kind):
    if kind == "brats128":
        import deepwmh_b200
        return deepwmh_b200.benchmark_plans(num_modalities=4, num_classes=4)
    return _plans(kind, 4, 4)                     # plans['num_classes'] = 3 labels; the network has 3 region outputs


def _region_pair(kind="cube", R_=3, seed=1, base=32, act="fp16", max_batch=8, M=4):
    """(plans, oracle network with sigmoid outputs, device trainer)."""
    import deepwmh_b200
    plans = _brats_plans(kind) if (M, base) == (4, 32) else _plans(kind, M, R_ + 1, base)
    net = RO.build_region_network(plans, seed, R_)

    class SigmoidTrainer(deepwmh_b200.nnUNetTrainerV2BraTSRegions):       # R_ sigmoid outputs
        def process_plans(self, plans):
            super().process_plans(plans)
            self.num_classes = R_

    tr = SigmoidTrainer(plans, device=0, act_dtype=act, max_batch=max_batch)
    tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
    assert tr.network.num_classes == R_ and tr.network.inference_nonlin == "sigmoid"
    return plans, net, tr


@pytest.mark.parametrize("kind", ["cube", "aniso", "brats128"])
def test_forward_patches_match_oracle_and_cuda_core(kind):
    plans, net, tr = _region_pair(kind)
    dev = tr.network
    n = 2 if kind == "brats128" else 4
    x = _patches(n, 4, dev.patch_size, seed=11)
    ref_dev = "cuda" if kind == "brats128" else "cpu"               # the 128^3 oracle runs on the GPU in fp32, TF32 off
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            ref = torch.sigmoid(net.float().to(ref_dev)(x.to(ref_dev))).cpu().numpy()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
        net.cpu()
    got = dev.forward_patches(x.cuda()).cpu().numpy()
    assert got.shape == (n, 3) + tuple(dev.patch_size)
    err = np.abs(got - ref).max()
    agree = np.mean((got > 0.5) == (ref > 0.5))
    inside = [float((ref[:, r] > 0.5).mean()) for r in range(3)]
    print("%s M=4 R=3  max |p - p_oracle| %.2e  region agreement %.5f  inside %s" % (kind, err, agree, inside))
    assert err < PROB_TOL and agree >= AGREE_MIN
    assert not np.allclose(got.sum(1), 1.0, atol=1e-3)                 # one sigmoid per output, not a softmax
    dev.set_force_generic(True)
    try:
        gen = dev.forward_patches(x.cuda()).cpu().numpy()
    finally:
        dev.set_force_generic(False)
    assert np.abs(gen - got).max() < PROB_TOL / 2, np.abs(gen - got).max()
    dev.close()


def sigmoid_head_report(w, last, probs):
    """max |p_dev - p_ref| / tol of the sigmoid head fed the device's own last-layer output `last` (float64), and the
    negative checks: the median of |p_swapped - p_ref| / tol over the last output (a coefficient chunk off by one) and the
    max of |softmax - p_ref| / tol.  A sigmoid passes an error of its logit on with a slope of at most 1/4, so the logit
    bound of head_report (1e-6 + 2^-14 sum_c |w_kc x_c|, here per output) bounds the probability error too."""
    p_ref = torch.sigmoid(F.conv3d(last, w))
    tol = 1e-6 + 2.0 ** -14 * F.conv3d(last.abs(), w.abs())
    err = ((probs - p_ref).abs() / tol).max().item()
    p_swap = torch.sigmoid(F.conv3d(last, swap_last_class_chunks(w)))
    sens_swap = torch.median(_sub((p_swap - p_ref)[:, -1:].abs() / tol[:, -1:])).item()
    sens_softmax = ((torch.softmax(F.conv3d(last, w), 1) - p_ref).abs() / tol).max().item()
    return err, sens_swap, sens_softmax


# (kind, outputs, base, act): three regions in both activation types and plans; every other output count on the cube;
# base 64 gives the head's one-voxel branch
HEAD_CASES = [("cube", 3, 32, "fp16"), ("aniso", 3, 32, "fp16"), ("cube", 3, 32, "bf16"), ("brats128", 3, 32, "fp16"),
              ("cube", 2, 32, "fp16"), ("cube", 4, 32, "fp16"), ("cube", 5, 32, "fp16"), ("cube", 6, 32, "fp16"),
              ("cube", 7, 32, "fp16"), ("cube", 8, 32, "fp16"), ("cube", 3, 64, "fp16"), ("cube", 8, 64, "bf16")]


@pytest.mark.parametrize("kind,R_,base,act", HEAD_CASES, ids=["%s-R%d-base%d-%s" % c for c in HEAD_CASES])
def test_sigmoid_head_matches_fp64_on_the_device_last_layer(kind, R_, base, act):
    M = 4 if base == 32 else 1
    plans, net, tr = _region_pair(kind, R_, base=base, act=act, M=M)
    dev = tr.network
    n = 2
    x = _patches(n, M, dev.patch_size, seed=3 + R_).cuda()
    probs = dev.forward_patches(x).double()
    last = dev.layer_output(dev.num_layers() - 1, n).double()
    w = net.seg_outputs[-1].weight.detach().to("cuda", torch.float64)
    err, sens_swap, sens_softmax = sigmoid_head_report(w, last, probs)
    print("%s R=%d base %d %s: sigmoid head max err/tol %.3f  swapped chunk %.1f  softmax %.1f"
          % (kind, R_, base, act, err, sens_swap, sens_softmax))
    assert err <= 1.0
    assert sens_swap >= SENS_MIN and sens_softmax > 1.0
    dev.close()


def _restated_overlap_add(rec):
    """The reference's tile loop in float32 fed the device's forwards: result += 1/n * unflip(p) per mirror (exact: n is a
    power of two), result *= gaussian (one rounding), agg[tile] += result (one rounding), nb[tile] += gaussian."""
    g = rec.g.float()
    agg = torch.zeros((rec.nw.num_classes,) + rec.shape, dtype=torch.float32, device="cuda")
    wgt = torch.zeros(rec.shape, dtype=torch.float32, device="cuda")
    nm = len(rec.mirrors)
    for t, parts in sorted(rec.probs.items()):
        for p in parts:
            p = p.float()
            r = torch.zeros((rec.nw.num_classes,) + rec.ps, dtype=torch.float32, device="cuda")
            for j, m in enumerate(rec.mirrors):
                dims = TT.flip_dims(m, 1)
                r = r + (1.0 / nm) * (p[j].flip(dims) if dims else p[j])
            r = r * g
            a = rec.tile(agg, t)
            a.copy_(a + r)
            wv = rec.tile(wgt, t)
            wv.copy_(wv + g)
    return agg, wgt


@pytest.mark.parametrize("kind,shape,mirror_axes,max_batch", [
    ("cube", (40, 50, 45), (0, 1, 2), 8), ("cube", (40, 50, 45), (0, 1), 8), ("cube", (35, 33, 37), (0, 1, 2), 16),
    ("aniso", (24, 70, 60), (0, 1, 2), 8)])
def test_region_overlap_add_is_the_reference_rounding_bit_for_bit(kind, shape, mirror_axes, max_batch):
    plans, net, tr = _region_pair(kind, max_batch=max_batch)
    dev = tr.network
    vol = torch.from_numpy(TT._volume_np(shape, 4, seed=5)).cuda()
    agg = torch.zeros((3,) + shape, device="cuda")
    wgt = torch.zeros(shape, device="cuda")
    dev.accumulate_tiles(vol, agg, wgt, 0.5, True, mirror_axes, True)
    rec = TT.Reconstruction(dev, vol, 0.5, True, mirror_axes, True, max_batch)
    agg_r, wgt_r = _restated_overlap_add(rec)
    bad = int((agg != agg_r).sum().item())
    print("%s %s mirrors %s mb%d: tiles %d, %d of %d sums differ from the float32 restatement"
          % (kind, "x".join(map(str, shape)), mirror_axes, max_batch, len(rec.origins), bad, agg.numel()))
    assert len(rec.origins) > 1 and bad == 0 and torch.equal(wgt, wgt_r)
    _, p = dev.finalize(agg, wgt, labels=False)
    assert torch.equal(p, agg_r / wgt_r)
    dev.close()


def test_region_labels_are_numpys_rule_bit_for_bit():
    plans, net, tr = _region_pair("cube")
    dev = tr.network
    shape = (37, 41, 29)                                          # V % 4 != 0
    vol = torch.from_numpy(TT._volume_np(shape, 4, seed=8)).cuda()
    _, p = dev.predict_3D(vol, True, use_sliding_window=True, step_size=0.5, use_gaussian=True, return_device_tensors=True)
    p = p.contiguous().clone()
    rng = np.random.default_rng(4)
    pn = p.cpu().numpy()
    half = np.float32(0.5)
    for val, frac in ((half, 0.05), (np.nextafter(half, np.float32(1)), 0.05), (np.nextafter(half, np.float32(0)), 0.05),
                      (np.float32(np.nan), 0.01)):
        pn[rng.random(pn.shape) < frac] = val
    pd = torch.from_numpy(pn).cuda()
    for order in ((1, 2, 3), (3, 1, 2), (255, 0, 7)):
        got = dev.region_labels(pd, order).cpu().numpy()
        want = RO.region_labels(pn, order)
        assert got.dtype == np.uint8 and np.array_equal(got.astype(np.float32), want), order
    # fewer regions than outputs is refused by the binding; one region on a plane of its own works
    with pytest.raises(ValueError):
        dev.region_labels(pd, (1, 2))
    one = pd[:1].contiguous()
    assert np.array_equal(dev.region_labels(one, (9,)).cpu().numpy().astype(np.float32), RO.region_labels(pn[:1], (9,)))
    dev.close()


# seeds whose random-init networks put every label on a fair share of the volume
@pytest.mark.parametrize("kind,shape,seed", [("cube", (50, 45, 41), 3), ("aniso", (30, 70, 60), 6)])
def test_tiled_predict_3d_with_tta_matches_oracle(kind, shape, seed):
    plans, net, tr = _region_pair(kind, seed=seed, max_batch=16)
    dev = tr.network
    x = TT._volume_np(shape, 4, seed=1)
    seg, p = tr.predict_preprocessed_data_return_seg_and_softmax(x, do_mirroring=True)
    seg_r, p_r = RO.OracleRegionTrainer(plans, net.float()).predict_preprocessed_data_return_seg_and_softmax(x, do_mirroring=True)
    assert p.shape == (3,) + shape and seg.shape == shape and seg.dtype == np.float32 == seg_r.dtype
    err, agree = np.abs(p - p_r).max(), np.mean(seg == seg_r)
    inside = [float((p_r[r] > 0.5).mean()) for r in range(3)]
    labels = [float((seg_r == c).mean()) for c in range(4)]
    print("%s predict_3D regions: max |p - p_oracle| %.2e  label agreement %.5f  inside %s  labels %s"
          % (kind, err, agree, inside, labels))
    assert all(0.05 < f < 0.95 for f in inside) and min(labels) > 0.02, (inside, labels)     # the agreement is not vacuous
    assert err <= 1e-2 and agree >= 0.998
    assert np.array_equal(seg, RO.region_labels(p, ORDER))
    # upstream's regions_class_order=None on a sigmoid network: the argmax; device tensors: uint8 labels
    seg_a, p_a = dev.predict_3D(x, True, use_sliding_window=True, step_size=0.5, use_gaussian=True)
    assert np.array_equal(p_a, p) and np.array_equal(seg_a, p.argmax(0))
    seg_d, p_d = dev.predict_3D(torch.from_numpy(x).cuda(), True, use_sliding_window=True, step_size=0.5, use_gaussian=True,
                                regions_class_order=ORDER, return_device_tensors=True)
    assert seg_d.dtype == torch.uint8 and np.array_equal(seg_d.cpu().numpy().astype(np.float32), seg)
    dev.close()


def test_softmax_network_refuses_regions_class_order():
    import deepwmh_b200
    plans = _plans("cube", 4, 4)
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0)
    tr.load_checkpoint_ram({"state_dict": O.build_benchmark_network(0, plans).state_dict()}, False)
    with pytest.raises(NotImplementedError, match="needs a sigmoid network"):
        tr.network.predict_3D(np.zeros((4, 32, 32, 32), np.float32), True, use_sliding_window=True, regions_class_order=ORDER)
    tr.network.close()


@pytest.mark.parametrize("kind", ["cube", "aniso"])
def test_bit_identical_repeat_and_split_tile_ranges(kind):
    plans, net, tr = _region_pair(kind)
    dev = tr.network
    shp = (48, 40, 40) if kind == "cube" else (24, 70, 60)
    vol = torch.from_numpy(np.random.default_rng(5).normal(size=(4,) + shp).astype(np.float32)).cuda()

    def run(ranges):
        agg = torch.zeros((3,) + shp, device="cuda")
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


def test_nnunet_predict_brats_regions_end_to_end(tmp_path, monkeypatch):
    """Four modalities through `nnUNet_predict -tr nnUNetTrainerV2BraTSRegions` with a spacing resample and a
    postprocessing.json, against crop -> resample -> z-score -> oracle region predict -> resample back -> region rule ->
    paste back -> largest component per entry."""
    from deepwmh_b200 import nifti, nnunet_predict as NP, preprocess
    from test_host_regions import _model_dir
    M = 4
    plans = _plans("cube", M, 4)
    plans["plans_per_stage"][0]["current_spacing"] = np.array([1.2, 1.0, 1.0])
    net = RO.build_region_network(plans, 3)
    root = str(tmp_path / "model")
    tdir = _model_dir(root, plans, "nnUNetTrainerV2BraTSRegions", net.state_dict())
    pp = {"for_which_classes": [[1, 2, 3], 3]}
    with open(os.path.join(tdir, "postprocessing.json"), "w") as f:
        json.dump(pp, f)
    vols = []
    for m in range(M):
        v = np.zeros((30, 44, 40), np.float32)
        v[2:28, 3:41, 4:37] = O.synthetic_flair((26, 38, 33), seed=60 + m)[0] * (1.0 + 0.3 * m)
        vols.append(v)
    indir = tmp_path / "in"; indir.mkdir()
    hdr = nifti.default_header((40, 44, 30), spacing=(1.0, 1.0, 1.1))
    for m in range(M):
        nifti.write_nifti(str(indir / ("caseT_%04d.nii.gz" % m)), np.transpose(vols[m], (2, 1, 0)), hdr)
    monkeypatch.setenv("RESULTS_FOLDER", root)
    out = str(tmp_path / "out")
    argv = ["-i", str(indir), "-o", out, "-t", "Task001_BrainTumour", "-tr", "nnUNetTrainerV2BraTSRegions", "-f", "all",
            "-chk", "model_best"]
    assert NP.main(argv) == 0
    assert json.load(open(os.path.join(out, "postprocessing.json"))) == pp
    seg = np.transpose(nifti.read_nifti(os.path.join(out, "caseT.nii.gz"))[0], (2, 1, 0))
    # oracle pipeline
    data = np.stack(vols)
    spacing = np.array([1.1, 1.0, 1.0])
    cropped, cseg, bbox = preprocess.crop_to_nonzero(data)
    target = np.array(plans["plans_per_stage"][0]["current_spacing"])
    d, _ = R.resample_and_normalize(cropped, cseg, spacing, target, True)
    _, p = RO.OracleRegionTrainer(plans, net.float()).predict_preprocessed_data_return_seg_and_softmax(d.astype(np.float32))
    p = R.resample_softmax_back(p, cropped.shape[1:], spacing, target)
    raw = preprocess.paste_back(RO.region_labels(p, ORDER).astype(np.uint8), data.shape[1:], bbox)
    ref = PO.remove_all_but_the_largest_connected_component(raw, [(1, 2, 3), 3], float(np.prod(hdr["spacing"])))
    agree = np.mean(seg == ref)
    labels = [float((ref == c).mean()) for c in range(4)]
    print("nnUNet_predict BraTS regions M=4: label agreement %.5f, label fractions %s" % (agree, labels))
    assert seg.max() <= 3 and agree > 0.997
    assert all(f > 0.001 for f in labels[1:]), labels
