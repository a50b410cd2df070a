"""Golden fixtures produced by the REFERENCE'S OWN in-tree code (run once in the authoring container, where
/root/reference is mounted; the GPU box never reads it).

The arithmetic either side of the network -- z_score, remove_sparks / remove_3mm_sparks, the stage-2 softmax masking
and checkpoint ensembling, the stage-1 NLL anomaly map pieces (group_mean / group_std / nll / mean_std_grid /
median_3mm / component_filtering) and the Dice of analysis/metrics.py -- lives in /root/reference itself, so unlike the un-vendored nnU-Net
engine these rows CAN be pinned: this script imports

    deepwmh/analysis/image_ops.py, deepwmh/analysis/lesion_analysis.py, deepwmh/pipeline/DCNN_multistage.py

unmodified (third-party modules that are absent here and not touched by these functions -- nibabel, skimage,
matplotlib, ... -- are replaced by inert stand-ins; NIfTI file access of the two stage-2 workers is redirected to an
in-memory dict) and stores their outputs on seeded inputs in tests/golden/intree_v1.npz.  The seeded inputs come from
tests/golden/fixtures.py, which also writes the file (inputs as digests; volumes the tests compare with a tolerance on
a fixed voxel sample).

usage: python tests/golden/make_golden_intree.py                 -> intree_v1.npz
       python tests/golden/make_golden_intree.py nll_analysis    -> nll_analysis_v1.npz (the whole nll_analysis, end to end)
"""
import os
import sys
from unittest.mock import MagicMock

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from golden import fixtures as F  # noqa: E402

REF = os.environ.get("DEEPWMH_REFERENCE", "DeepWMH")          # a checkout of the original DeepWMH project
SAMPLED_INTREE = ["zscore_plain", "group_mean", "group_std", "nll_none", "nll_neg", "nll_mu", "nll_sigma", "nll_eps",
                  "pipe_x_prime", "pipe_local_mu", "pipe_anomaly", "pipe_mean", "pipe_std", "pipe_ref_anomaly0", "pipe_anomaly_cf",
                  "group_mean_masked", "group_std_masked", "nll_usemask", "nll_usemask_mu", "nll_usemask_sigma"] + \
                 ["msg_%s_%s" % (a, t) for t in ("p12", "p50", "podd", "nomask") for a in ("mean", "std")]
SAMPLED_NLL = ["%s_%s" % (n, t) for t in ("pos", "none") for n in ("normalized_input", "intensity_thr", "local_mean", "mean_value", "std_value")]


def import_reference():
    sys.path.insert(0, REF)
    stubbed = []
    for _ in range(64):
        try:
            import deepwmh.analysis.image_ops as io
            import deepwmh.analysis.lesion_analysis as la
            import deepwmh.analysis.metrics as mt
            import deepwmh.pipeline.DCNN_multistage as ms
            return io, la, mt, ms, stubbed
        except ModuleNotFoundError as e:
            m = MagicMock()
            m.__path__, m.__name__, m.__spec__ = [], e.name, None
            sys.modules[e.name] = m
            stubbed.append(e.name)
    raise RuntimeError("could not import the reference")


def main():
    io, la, mt, ms, stubbed = import_reference()
    out = {"stubbed_modules": np.array(stubbed)}
    inp = F.intree_inputs()

    # ---- z_score / masked_mean / masked_std (image_ops.py:13-21,172-179)
    target, refs, brain, valid = inp["in_target"], list(inp["in_refs"]), inp["in_brain"], inp["in_valid"]
    out["in_target"], out["in_refs"], out["in_brain"], out["in_valid"] = target, np.stack(refs), brain, valid
    out["zscore_masked"] = io.z_score(target, mask=brain)
    out["zscore_plain"] = io.z_score(target)
    out["masked_mean_std"] = np.array([io.masked_mean(target, brain), io.masked_std(target, brain)], dtype=np.float64)

    # ---- remove_sparks / remove_3mm_sparks (image_ops.py:325-367)
    sp = inp["sparks_in"]
    out["sparks_in"] = sp
    for name, vox in (("iso1", [1.0, 1.0, 1.0]), ("iso05", [0.5, 0.5, 0.5]), ("iso2", [2.0, 2.0, 2.0]),
                      ("thick", [1.0, 1.0, 6.0]), ("aniso", [0.9, 0.9, 2.5])):
        out["sparks_" + name] = io.remove_3mm_sparks(sp, vox).astype(np.uint8)
        out["sparks_vox_" + name] = np.array(vox)
    out["sparks_min5"] = io.remove_sparks(sp, min_volume=5).astype(np.uint8)

    # ---- stage-2 masking + ensembling workers (DCNN_multistage.py:102-125), NIfTI access redirected to memory.
    # load_nifti_simple returns float32 (utilities/data_io.py), save_nifti stores what it is given.
    store = {}
    ms.load_nifti_simple = lambda p: np.asarray(store[p]).astype("float32")
    ms.save_nifti = lambda data, hdr, p: store.__setitem__(p, np.asarray(data))
    ms.get_nifti_header = lambda p: None
    ms.try_load_nifti = lambda p: False
    ms.file_exist = lambda p: False
    shape = (33, 40, 29)
    xs, m = list(inp["ens_x"]), inp["ens_mask"]
    store["mask"] = m
    masked = []
    for i, x in enumerate(xs):
        store["x%d" % i] = x
        ms._parallel_softmax_masking(("x%d" % i, "mask", "y%d" % i))
        masked.append("y%d" % i)
    ms._parallel_ensembling((masked, None, None, "field", "label", shape, [1.0, 1.0, 1.0]))
    out["ens_x"], out["ens_mask"] = np.stack(xs), m
    out["ens_field"], out["ens_label"] = store["field"], store["label"].astype(np.uint8)
    out["ens_y0_dtype"] = np.array(str(store["y0"].dtype))

    # ---- Dice (analysis/metrics.py:26-32)
    a, b = inp["dice_in"]
    dice_fn = [getattr(mt, n) for n in dir(mt) if "dice" in n.lower() and callable(getattr(mt, n))]
    out["dice_in"] = np.stack([a, b])
    out["dice_names"] = np.array([f.__name__ for f in dice_fn])
    vals = []
    for f in dice_fn:
        try:
            vals.append(float(f(a, b)))
        except Exception:
            vals.append(np.nan)
    out["dice_vals"] = np.array(vals)

    # ---- stage-1 pieces (lesion_analysis.py:84-113; image_ops.py:56-170,197-231,378-421)
    # the isolated pieces consume fp32-rounded inputs (what the device kernels are handed), so that they and the
    # reference see identical numbers; the composed pipeline further down stays float64 end to end as in the reference
    zt = io.z_score(target, mask=brain).astype("float32")
    zr = [io.z_score(r, mask=brain).astype("float32") for r in refs]
    out["z_target"], out["z_refs"] = zt, np.stack(zr)
    out["group_mean"] = io.group_mean(zr)
    out["group_std"] = io.group_std(zr)
    for side, tag in ((None, "none"), ("+", "pos"), ("-", "neg")):
        an, mu, sg = la.nll(zt, zr, min_std=0.03, side=side, return_all=True)
        out["nll_" + tag] = an
    out["nll_mu"], out["nll_sigma"] = mu, sg
    out["nll_eps"] = la.nll(zt, zr, min_std=None, side=None)
    for ps, tag in (([12, 12, 12], "p12"), ([50, 50, 50], "p50"), ([9, 14, 11], "podd")):
        mi, si = io.mean_std_grid(zt, ps, mask=valid)
        out["msg_mean_" + tag], out["msg_std_" + tag] = mi, si
        out["msg_patch_" + tag] = np.array(ps)
    mi, si = io.mean_std_grid(zt, [12, 12, 12])
    out["msg_mean_nomask"], out["msg_std_nomask"] = mi, si
    an = out["nll_pos"].astype("float32")
    for vox, tag in (([1.0, 1.0, 1.0], "iso1"), ([0.7, 0.7, 0.7], "iso07"), ([0.5, 0.6, 1.5], "mixed"),
                     ([0.9, 0.9, 5.0], "thick")):
        out["median_" + tag] = io.median_3mm(an, vox)
        out["median_vox_" + tag] = np.array(vox)

    # ---- the array part of nll_analysis (lesion_analysis.py:150-181), composed from the reference functions exactly
    # as written there (apply_otsu=False: skimage is absent here; component_filtering left out: host-side mask work).
    patch = [14, 14, 14]
    x_prime = io.z_score(target, mask=brain)
    tissue_min = np.ma.masked_array(x_prime, mask=1 - brain).min()
    x_prime = np.where(brain < 0.5, tissue_min, x_prime)
    x_i = []
    for r in refs:
        t = io.z_score(r, mask=brain)
        tmin = np.ma.masked_array(t, mask=1 - brain).min()
        x_i.append(np.where(brain < 0.5, tmin, t))
    mu_p, _ = io.mean_std_grid(x_prime, patch, mask=valid)
    for i in range(len(x_i)):
        mu_i, _ = io.mean_std_grid(x_i[i], patch, mask=valid)
        x_i[i] = x_i[i] - mu_i + mu_p
    an, xm, xs_ = la.nll(x_prime, x_i, min_std=0.03, side="+", return_all=True)
    out["pipe_patch"] = np.array(patch)
    out["pipe_x_prime"], out["pipe_local_mu"] = x_prime, mu_p
    out["pipe_anomaly"], out["pipe_mean"], out["pipe_std"] = an * valid, xm, xs_
    out["pipe_ref_anomaly0"] = la.nll(x_i[0], x_i, min_std=0.03, side="+") * valid

    # ---- component_filtering (image_ops.py:253-306): per-slice erosion + largest component, three orientations
    speck = inp["cf_in"]                                            # the valid mask plus sparks outside the brain
    out["cf_in"] = speck
    for vox, tag in (([1.0, 1.0, 1.0], "iso"), ([0.9, 0.9, 4.0], "thick_z"), ([5.0, 1.0, 1.0], "thick_x")):
        out["cf_" + tag] = io.component_filtering(speck, vox).astype(np.float32)
        out["cf_vox_" + tag] = np.array(vox)
    out["cf_brain"] = io.component_filtering(brain, [1.0, 1.0, 1.0]).astype(np.float32)
    out["cf_empty"] = io.component_filtering(np.zeros((6, 7, 5), "float32"), [1.0, 1.0, 1.0]).astype(np.float32)
    out["pipe_anomaly_cf"] = an * valid * io.component_filtering(valid, [1.0, 1.0, 1.0])      # lesion_analysis.py:175-176

    # ---- group_mean / group_std with masks (image_ops.py:197-231) and the Otsu branch of nll (lesion_analysis.py:87-92).
    # skimage is absent, so for nll(use_mask=True) the restated threshold_otsu (oracle/intree_oracle.py, unpinned) is
    # injected into the reference module; everything else on that path is the reference's own code.
    gm = list(inp["gmask"])                                         # with a slab no reference covers -> NaN
    out["gmask"] = np.stack(gm)
    out["group_mean_masked"] = io.group_mean(zr, masks=gm)
    out["group_std_masked"] = io.group_std(zr, masks=gm)
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import intree_oracle as I
    la.threshold_otsu = I.threshold_otsu
    an, mu, sg = la.nll(zt, zr, min_std=0.03, side="+", return_all=True, use_mask=True)
    out["nll_usemask"], out["nll_usemask_mu"], out["nll_usemask_sigma"] = an, mu, sg

    conv = {}
    for k_, v in out.items():
        v = np.asarray(v)
        conv[k_] = v.astype(np.float32) if v.dtype == np.float64 and v.ndim >= 3 else v   # volumes: fp32 on disk
    F.save(os.path.join(HERE, "intree_v1.npz"), {k: v for k, v in conv.items() if k not in inp}, {k: conv[k] for k in inp}, SAMPLED_INTREE)
    print("wrote intree_v1.npz:", len(conv), "arrays;", "stubbed:", ", ".join(stubbed))


if __name__ == "__main__" and "nll_analysis" not in sys.argv[1:]:
    main()


def nll_analysis_fixture():
    """Run the reference's nll_analysis (lesion_analysis.py:115-281) END TO END, unmodified, on seeded in-memory volumes:
    its NIfTI readers / writers are redirected to a dict, the plot is a no-op, apply_otsu=False (skimage is absent).
    -> tests/golden/nll_analysis_v1.npz"""
    io, la, mt, ms, stubbed = import_reference()
    inp = F.nll_analysis_inputs()
    k = len(inp["in_refs"])
    store = {"x": inp["in_target"]}
    for i in range(k):
        store["r%d" % i], store["m%d" % i], store["y%d" % i] = inp["in_refs"][i], inp["in_label1"][i], inp["in_label2"][i].astype("float32")
    vox = (1.0, 1.2, 1.1)
    la.get_nifti_pixdim = lambda p: list(vox)
    la.load_nifti_simple = lambda p: np.asarray(store[p]).astype("float32")
    la.load_nifti = lambda p: (np.asarray(store[p]).astype("float32"), None)
    la.save_nifti = lambda data, hdr, p: store.__setitem__("out:" + os.path.basename(p), np.asarray(data))
    la.hist_plot = lambda *a, **kw: None
    la.mkdir = lambda p: p
    case = {"x": "x", "r": ["r%d" % i for i in range(k)], "m": ["m%d" % i for i in range(k)], "y": ["y%d" % i for i in range(k)]}
    out = {"voxel_size": np.array(vox)}
    for prior, tag in (("+", "pos"), (None, "none")):
        an, valid, cx, cy, cr, thr = la.nll_analysis(case, apply_otsu=False, intensity_prior=prior, case_output_folder="o", debug=True)
        out["anomaly_" + tag], out["valid_" + tag] = np.asarray(an, np.float32), np.asarray(valid, np.float32)
        out["curve_x_" + tag], out["curve_y_" + tag], out["curve_r_" + tag] = cx, cy, cr
        out["threshold_" + tag] = np.array(thr)
        for name in ("normalized_input", "intensity_thr", "rough_brain", "local_mean", "mean_value", "std_value", "averaged_label"):
            out[name + "_" + tag] = np.asarray(store["out:" + name + ".nii.gz"], np.float32)
    F.save(os.path.join(HERE, "nll_analysis_v1.npz"), out, inp, SAMPLED_NLL)
    print("wrote nll_analysis_v1.npz:", {k_: (v.shape if hasattr(v, "shape") else v) for k_, v in out.items() if k_.startswith(("thr", "curve_x"))})


if __name__ == "__main__" and "nll_analysis" in sys.argv[1:]:
    nll_analysis_fixture()
