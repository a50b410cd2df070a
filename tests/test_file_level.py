"""File-level drop-in (SURVEY.md section 8 rows a1, f-1, f-2): NIfTI I/O, nnU-Net cropping / paste-back, 3 mm spark
removal, model-directory discovery, and the DeepWMH_predict-compatible command line."""
import gzip
import os
import pickle
import struct

import numpy as np
import pytest
import torch
from scipy.ndimage import binary_fill_holes, label

import oracle as O
from conftest import small_plans
from deepwmh_b200 import cli, nifti, preprocess
from golden.fixtures import intree as intree_fixture


def test_nifti_round_trip_and_header(tmp_path):
    rng = np.random.default_rng(0)
    vol = rng.normal(size=(7, 9, 5)).astype(np.float32)
    hdr = nifti.default_header(vol.shape, spacing=(0.9, 1.1, 3.0))
    for name in ("a.nii", "a.nii.gz"):
        p = str(tmp_path / name)
        nifti.write_nifti(p, vol, hdr)
        back, h2 = nifti.read_nifti(p)
        assert back.dtype == np.float32 and np.array_equal(back, vol)
        assert np.allclose(h2["spacing"], (0.9, 1.1, 3.0)) and h2["shape"] == (7, 9, 5)
    raw = gzip.open(str(tmp_path / "a.nii.gz"), "rb").read()
    assert struct.unpack("<i", raw[:4])[0] == 348 and raw[344:348] == b"n+1\x00"
    assert struct.unpack("<8h", raw[40:56])[:4] == (3, 7, 9, 5)
    # x is the fastest axis on disk (NIfTI / nibabel convention)
    first = np.frombuffer(raw, dtype="<f4", count=7, offset=352)
    assert np.array_equal(first, vol[:, 0, 0])
    # integer storage + scaling
    seg = (rng.random((7, 9, 5)) > 0.5).astype(np.uint8)
    nifti.write_nifti(str(tmp_path / "s.nii.gz"), seg, h2, dtype=np.uint8)
    b2, _ = nifti.read_nifti(str(tmp_path / "s.nii.gz"))
    assert np.array_equal(b2, seg.astype(np.float32))
    raw = bytearray(gzip.open(str(tmp_path / "s.nii.gz"), "rb").read())
    struct.pack_into("<ff", raw, 112, 2.0, 1.0)                  # scl_slope, scl_inter
    open(str(tmp_path / "t.nii"), "wb").write(bytes(raw))
    b3, _ = nifti.read_nifti(str(tmp_path / "t.nii"))
    assert np.array_equal(b3, seg.astype(np.float32) * 2 + 1)
    with pytest.raises(ValueError):
        open(str(tmp_path / "bad.nii"), "wb").write(b"\x00" * 400)
        nifti.read_nifti(str(tmp_path / "bad.nii"))


def test_crop_to_nonzero_and_paste_back():
    rng = np.random.default_rng(1)
    data = np.zeros((1, 20, 24, 22), np.float32)
    data[0, 3:15, 5:20, 2:18] = rng.normal(5, 1, size=(12, 15, 16))
    data[0, 7:9, 9:12, 6:9] = 0                                   # a hole: filled in the mask, so seg stays 0 there
    cropped, seg, bbox = preprocess.crop_to_nonzero(data)
    assert bbox == [[3, 15], [5, 20], [2, 18]] and cropped.shape == (1, 12, 15, 16) and seg.shape == (1, 12, 15, 16)
    ref_mask = binary_fill_holes(data[0] != 0)[3:15, 5:20, 2:18]
    assert np.array_equal(seg[0] >= 0, ref_mask) and (seg[0][4:6, 4:7, 4:7] == 0).all()
    pred = (rng.random((12, 15, 16)) > 0.5).astype(np.uint8)
    full = preprocess.paste_back(pred, data.shape[1:], bbox)
    assert full.shape == (20, 24, 22) and np.array_equal(full[3:15, 5:20, 2:18], pred) and full.sum() == pred.sum()
    empty = np.zeros((1, 4, 4, 4), np.float32)
    c2, s2, b2 = preprocess.crop_to_nonzero(empty)
    assert c2.shape == empty.shape and (s2 == -1).all()


def test_remove_3mm_sparks_matches_reference_algorithm():
    rng = np.random.default_rng(2)
    m = (rng.random((24, 24, 24)) > 0.82).astype(np.float32)

    def ref(mask, min_volume):                                    # the loop of analysis/image_ops.py:325-344
        lab, n = label((mask > 0.5).astype("int"))
        out = np.zeros_like(lab)
        for i in range(1, n + 1):
            if (lab == i).sum() >= min_volume:
                out[lab == i] = 1
        return out
    assert np.array_equal(preprocess.remove_3mm_sparks(m, [1.0, 1.0, 1.0]), ref(m, 3))
    assert np.array_equal(preprocess.remove_3mm_sparks(m, [0.5, 0.5, 0.5]), ref(m, 24))
    assert np.array_equal(preprocess.remove_3mm_sparks(m, [2.0, 2.0, 2.0]), ref(m, 2))        # round(3/8)=0 -> 2
    assert np.array_equal(preprocess.remove_3mm_sparks(m, [1.0, 1.0, 6.0]), ref(m, 3))        # thick slices
    assert preprocess.remove_3mm_sparks(np.zeros((4, 4, 4)), [1, 1, 1]).sum() == 0


def _make_model_dir(root, plans, net, task="Task002_FinalModel"):
    tdir = os.path.join(root, "nnUNet", "3d_fullres", task, "nnUNetTrainerV2__nnUNetPlansv2.1")
    os.makedirs(os.path.join(tdir, "all"))
    pickle.dump(plans, open(os.path.join(tdir, "plans.pkl"), "wb"))
    torch.save({"epoch": 1, "state_dict": net.state_dict()}, os.path.join(tdir, "all", "model_best.model"))
    pickle.dump({"init": (os.path.join(tdir, "plans.pkl"), "all", tdir, "", True, 0, True, False, True),
                 "name": "nnUNetTrainerV2", "class": "x", "plans": plans},
                open(os.path.join(tdir, "all", "model_best.model.pkl"), "wb"))
    return tdir


def test_model_directory_discovery(tmp_path):
    plans = small_plans()
    net = O.build_benchmark_network(0, plans)
    root = str(tmp_path / "model")
    _make_model_dir(root, plans, net)
    m = cli.find_model(root)
    assert m["task"] == "Task002_FinalModel" and os.path.isfile(m["plans"]) and os.path.isfile(m["checkpoint"])
    assert cli.load_plans(m["plans"])["base_num_features"] == 32
    with pytest.raises(RuntimeError, match="nnUNet"):
        cli.find_model(str(tmp_path))
    _make_model_dir(root, plans, net, task="Task003_Other")
    with pytest.raises(RuntimeError, match="multiple"):
        cli.find_model(root)
    assert cli.find_model(root, "Task003_Other")["task"] == "Task003_Other"


def test_cli_argument_errors(tmp_path):
    plans = small_plans()
    root = str(tmp_path / "model")
    _make_model_dir(root, plans, O.build_benchmark_network(0, plans))
    img = str(tmp_path / "a.nii.gz")
    nifti.write_nifti(img, np.ones((8, 8, 8), np.float32), nifti.default_header((8, 8, 8)))
    with pytest.raises(RuntimeError, match="should be equal"):
        cli.main(["-i", img, img, "-n", "a", "-m", root, "-o", str(tmp_path / "o"), "--skip-bfc"])
    with pytest.raises(SystemExit):
        cli.main(["-i", img, img, "-n", "a", "a", "-m", root, "-o", str(tmp_path / "o"), "--skip-bfc"])
    with pytest.raises(SystemExit):
        cli.main(["-i", str(tmp_path / "missing.nii.gz"), "-n", "a", "-m", root, "-o", str(tmp_path / "o"), "--skip-bfc"])
    with pytest.raises(RuntimeError, match="nnUNet"):
        cli.main(["-i", img, "-n", "a", "-m", str(tmp_path), "-o", str(tmp_path / "o"), "--skip-bfc"])


def test_robex_fov_masking_step(tmp_path):
    """predict.py:39-48,165-181 with a stand-in runROBEX.sh (the real one is an external program): seg x brain mask."""
    rng = np.random.default_rng(3)
    img_dir, d3, dfov, rb = (tmp_path / n for n in ("img", "p3", "fov", "robex"))
    for d in (img_dir, d3, dfov, rb):
        d.mkdir()
    hdr = nifti.default_header((10, 12, 8))
    seg = (rng.random((10, 12, 8)) > 0.6).astype(np.float32)
    mask = np.zeros((10, 12, 8), np.float32); mask[2:8, 3:9, 1:7] = 1
    nifti.write_nifti(str(img_dir / "c1_0000.nii.gz"), rng.normal(size=(10, 12, 8)).astype(np.float32), hdr)
    nifti.write_nifti(str(d3 / "c1.nii.gz"), seg, hdr, dtype=np.float32)
    nifti.write_nifti(str(rb / "mask_src.nii.gz"), mask, hdr, dtype=np.float32)
    with pytest.raises(RuntimeError, match="ROBEX"):
        cli.robex_fov_masking(["c1"], str(img_dir), str(d3), str(dfov), str(rb))          # binaries missing
    (rb / "ROBEX").write_text("")
    (rb / "runROBEX.sh").write_text("#!/bin/sh\ncp \"$1\" \"$2\"\ncp %s \"$3\"\n" % (rb / "mask_src.nii.gz"))
    os.chmod(str(rb / "runROBEX.sh"), 0o755)
    cli.robex_fov_masking(["c1"], str(img_dir), str(d3), str(dfov), str(rb))
    out, _ = nifti.read_nifti(str(dfov / "c1.nii.gz"))
    assert np.array_equal(out, ((seg * mask) > 0.5).astype(np.float32))
    assert sorted(os.listdir(str(dfov))) == ["c1.nii.gz"]                                   # temporaries removed


@pytest.mark.gpu
def test_cli_end_to_end_matches_oracle_pipeline(tmp_path):
    """DeepWMH_predict-style run on a tiny model: output tree, raw segmentation equal to the oracle run through the
    same crop / z-score / predict / paste-back steps, 3 mm post-processing file present."""
    plans = small_plans()
    plans["use_mask_for_norm"] = {0: True}
    net = O.build_benchmark_network(0, plans)
    root = str(tmp_path / "model")
    _make_model_dir(root, plans, net)
    vol_zyx = np.zeros((44, 52, 48), np.float32)
    vol_zyx[4:42, 6:50, 5:45] = O.synthetic_flair((38, 44, 40), seed=11)[0]
    vol_zyx[4:42, 6:50, 5:45][vol_zyx[4:42, 6:50, 5:45] == 0] = 3.0           # solid block: crop = the block
    img = str(tmp_path / "case1.nii.gz")
    nifti.write_nifti(img, np.transpose(vol_zyx, (2, 1, 0)), nifti.default_header((48, 52, 44)))
    out = str(tmp_path / "out")
    assert cli.main(["-i", img, "-n", "case1", "-m", root, "-o", out, "--skip-bfc", "-g", "0"]) == 0
    assert os.path.isfile(os.path.join(out, "001_Preprocessed_Images", "case1_0000.nii.gz"))
    seg_xyz, hdr = nifti.read_nifti(os.path.join(out, "002_Segmentations", "001_raw", "case1.nii.gz"))
    assert os.path.isfile(os.path.join(out, "002_Segmentations", "002_postproc_3mm", "case1.nii.gz"))
    seg = np.transpose(seg_xyz, (2, 1, 0))
    assert seg.shape == vol_zyx.shape and seg[:4].sum() == 0
    cropped, s, bbox = preprocess.crop_to_nonzero(vol_zyx[None])
    assert bbox == [[4, 42], [6, 50], [5, 45]]
    norm = O.zscore_nnunet(cropped[0], s[0], True)[None]
    seg_ref, _ = O.OracleTrainer(plans, net).predict_preprocessed_data_return_seg_and_softmax(norm)
    full_ref = preprocess.paste_back(seg_ref.astype(np.uint8), vol_zyx.shape, bbox)
    assert np.mean(full_ref == seg) > 0.998


@pytest.mark.gpu
def test_device_remove_sparks_matches_scipy_components():
    """SURVEY 8f-2: dwmh_remove_sparks (union-find CCL on the device) is bit-identical to the scipy.ndimage.label loop of
    image_ops.py:325-344, and remove_3mm_sparks applies the same voxel-size rule."""
    import deepwmh_b200
    plans = small_plans()
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=1)
    net = tr.network
    rng = np.random.default_rng(5)
    for shape, thr in (((24, 24, 24), 0.82), ((37, 19, 45), 0.7), ((64, 80, 48), 0.55), ((5, 7, 3), 0.5), ((1, 1, 9), 0.4)):
        m = (rng.random(shape) > thr).astype(np.uint8)
        m_dev = torch.from_numpy(m).cuda()
        for mv in (1, 2, 3, 24):
            got = net.remove_sparks(m_dev, mv).cpu().numpy()
            assert np.array_equal(got, preprocess.remove_sparks(m, mv).astype(np.uint8)), (shape, mv)
        for vs in ([1.0, 1.0, 1.0], [0.5, 0.5, 0.5], [2.0, 2.0, 2.0], [1.0, 1.0, 6.0]):
            got = net.remove_3mm_sparks(m_dev, vs).cpu().numpy()
            assert np.array_equal(got, preprocess.remove_3mm_sparks(m, vs).astype(np.uint8)), (shape, vs)
    z = torch.zeros((8, 8, 8), dtype=torch.uint8, device="cuda")
    assert net.remove_sparks(z, 3).sum().item() == 0
    o = torch.ones((8, 9, 10), dtype=torch.uint8, device="cuda")
    assert net.remove_sparks(o, 3).sum().item() == 720
    # a serpentine one-voxel-wide component exercises long union chains; labels > 1 in the input count as foreground
    s = np.zeros((16, 16, 16), np.uint8)
    for i in range(16):
        s[i, :, 0 if i % 2 == 0 else 15] = 2
        s[i, 15 if i % 2 == 0 else 0, :] = 2
    got = net.remove_sparks(torch.from_numpy(s).cuda(), 3).cpu().numpy()
    assert np.array_equal(got, preprocess.remove_sparks(s, 3).astype(np.uint8))
    # outputs of the reference's own remove_sparks / remove_3mm_sparks (tests/golden/make_golden_intree.py)
    g = intree_fixture()
    sp = torch.from_numpy((g["sparks_in"] > 0.5).astype(np.uint8)).cuda()
    for tag in ("iso1", "iso05", "iso2", "thick", "aniso"):
        got = net.remove_3mm_sparks(sp, g["sparks_vox_" + tag].tolist()).cpu().numpy()
        assert np.array_equal(got, g["sparks_" + tag]), tag
    assert np.array_equal(net.remove_sparks(sp, 5).cpu().numpy(), g["sparks_min5"])
    net.close()


def _ref_masked_ensemble(xs, m, voxel_size):
    """numpy restatement of _parallel_softmax_masking + _parallel_ensembling (DCNN_multistage.py:102-125): float32 arrays
    from load_nifti_simple (utilities/data_io.py:288-290), float32 running field; pinned by tests/test_intree_oracle.py."""
    from oracle import intree_oracle as I
    field, label = I.ensembling([I.softmax_masking(x, m) for x in xs], voxel_size)
    return field, label.astype(np.uint8)


@pytest.mark.gpu
def test_device_masked_ensemble_is_bit_exact():
    """SURVEY 8f-3: dwmh_ensemble_masked_add / dwmh_ensemble_refine reproduce the reference's masked checkpoint ensemble
    bit for bit on the same background-probability inputs."""
    import deepwmh_b200
    plans = small_plans()
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=1)
    net = tr.network
    rng = np.random.default_rng(9)
    shape = (33, 40, 29)
    xs = [np.clip(rng.normal(0.5, 0.35, size=shape), 0, 1).astype(np.float32) for _ in range(5)]
    xs[2][:4] = 0.5                                              # exact ties stay background (field < 0.5 is strict)
    m = (rng.random(shape) > 0.3).astype(np.float32)
    for mask in (m, None):
        acc = torch.zeros(shape, dtype=torch.float32, device="cuda")
        md = torch.from_numpy(mask).cuda() if mask is not None else None
        for x in xs:
            net.ensemble_masked_add_(acc, torch.from_numpy(x).cuda(), md)
        label = net.ensemble_refine_(acc, len(xs))
        clean = net.remove_3mm_sparks(label, [1.0, 1.0, 1.0])
        f_ref, l_ref = _ref_masked_ensemble(xs, mask if mask is not None else np.ones(shape, np.float32), [1.0, 1.0, 1.0])
        assert np.array_equal(acc.cpu().numpy(), f_ref)
        assert np.array_equal(clean.cpu().numpy(), l_ref)
    # the reference's own two workers on seeded inputs (tests/golden/make_golden_intree.py)
    g = intree_fixture()
    acc = torch.zeros(g["ens_field"].shape, dtype=torch.float32, device="cuda")
    md = torch.from_numpy(g["ens_mask"]).cuda()
    for x in g["ens_x"]:
        net.ensemble_masked_add_(acc, torch.from_numpy(x).cuda(), md)
    label = net.remove_3mm_sparks(net.ensemble_refine_(acc, len(g["ens_x"])), [1.0, 1.0, 1.0])
    assert np.array_equal(acc.cpu().numpy(), g["ens_field"]) and np.array_equal(label.cpu().numpy(), g["ens_label"])
    net.close()


@pytest.mark.gpu
def test_checkpoint_ensemble_refined_label_end_to_end():
    """The k-checkpoint loop (load_checkpoint_ram -> no-TTA prediction -> masked mean -> < 0.5 -> 3 mm sparks) against the
    same pipeline run with the oracle's predictions."""
    import deepwmh_b200
    from deepwmh_b200 import parallel
    plans = small_plans()
    nets = [O.build_benchmark_network(k, plans) for k in range(3)]
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=8)
    vol = O.synthetic_flair((40, 44, 36), seed=3)
    data = O.zscore_nnunet(vol[0], (vol[0] != 0).astype(np.int8) - 1, True)[None]
    m = (vol[0] != 0).astype(np.float32)
    field, label = parallel.checkpoint_ensemble_refined_label(tr, [{"state_dict": n.state_dict()} for n in nets], data, m, (1.0, 1.0, 1.0))
    xs = []
    for n in nets:
        _, sm = O.OracleTrainer(plans, n).predict_preprocessed_data_return_seg_and_softmax(data, do_mirroring=False)
        xs.append(sm[0].astype(np.float32))
    f_ref, l_ref = _ref_masked_ensemble(xs, m, [1.0, 1.0, 1.0])
    assert field.shape == f_ref.shape and label.dtype == torch.uint8
    assert np.abs(field.cpu().numpy() - f_ref).max() < 1e-2
    assert np.mean(label.cpu().numpy() == l_ref) > 0.995
    assert (field.cpu().numpy()[m == 0] == 1.0).all()           # outside the valid mask the field is exactly "background"
    tr.network.close()
