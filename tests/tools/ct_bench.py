"""Device time of the CT normalisation and cascade kernels, and one 512 x 512 x 300 CT case through nnUNet_predict's
3d_fullres, 3d_lowres and 3d_cascade_fullres (DESIGN §13) -> profiles/ct_r03.json.

  * dwmh_ct_normalize CT / CT2 at 182 x 218 x 182 (29 MB: L2-resident after the first pass, which a pass over the same
    volume keeps) and 512 x 512 x 320 (336 MB, above the 126 MB L2), CUDA events around `--iters` back-to-back calls after a
    warm-up; GB/s from the algorithmic bytes (CT: read + write, 8 B/voxel; CT2: two reads + one write, 12 B/voxel, its
    second read is served by L2 only below its size) against 7.7 TB/s.
  * dwmh_cascade_onehot: 256 x 256 x 160 labels onto 512 x 512 x 320, three classes (two fp32 planes written).
  * nnUNet_predict wall time of one int16 CT case (file read to label file written) with random-init 128^3-patch networks
    for 3d_fullres, 3d_lowres and 3d_cascade_fullres (its automatic low-resolution pass included), after a warm-up run of
    the cascade on a smaller crop of the case; --tta selects 8x mirroring (default off, see the json).
The card's name and power limit are read by the same process that times.  Needs a GPU; writes --out (default
profiles/ct_r03.json).
"""
import argparse
import json
import os
import pickle
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import oracle as O  # noqa: E402
from deepwmh_b200 import nifti, preprocess  # noqa: E402
from deepwmh_b200 import nnunet_predict as NP  # noqa: E402
from deepwmh_b200.plans import benchmark_plans  # noqa: E402

PEAK_TBS = 7.7
CT = {"mean": 80.0, "sd": 120.0, "percentile_00_5": -1000.0, "percentile_99_5": 1500.0}


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def _time(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3          # us per call


def kernels(iters):
    rows = []
    for shape, where in (((182, 218, 182), "L2-resident"), ((512, 512, 320), "above L2")):
        n = int(np.prod(shape))
        g = torch.Generator(device="cuda").manual_seed(0)
        v = (torch.rand(n, generator=g, device="cuda") * 3000 - 1200).contiguous()
        for scheme, bpv in (("CT", 8), ("CT2", 12)):
            c = CT if scheme == "CT" else {k: CT[k] for k in ("percentile_00_5", "percentile_99_5")}
            # CT2 is timed without its statistics read-back (no host synchronisation inside the loop)
            fn = (lambda: preprocess.ct_normalize_device(v, None, "CT", c)) if scheme == "CT" else (lambda: _ct2_nosync(v, c))
            us = _time(fn, iters)
            gbs = bpv * n / (us * 1e-6) / 1e9
            rows.append({"kernel": scheme, "shape": list(shape), "working_set": where, "device_us": round(us, 2),
                         "algorithmic_GB_per_s": round(gbs, 1), "share_of_7.7_TB_per_s": round(gbs / (PEAK_TBS * 1e3), 3),
                         "bytes_per_voxel": bpv, "status": "measured"})
    lab = torch.randint(0, 3, (256, 256, 160), dtype=torch.uint8, device="cuda")
    out = torch.empty((2, 512, 512, 320), dtype=torch.float32, device="cuda")
    us = _time(lambda: preprocess.cascade_onehot_device(lab, out, 3), iters)
    wb = out.numel() * 4
    rows.append({"kernel": "cascade_onehot", "shape": [256, 256, 160], "out_shape": [512, 512, 320], "num_classes": 3,
                 "device_us": round(us, 2), "written_GB_per_s": round(wb / (us * 1e-6) / 1e9, 1), "status": "measured"})
    return rows


_WS = {}


def _ct2_nosync(v, c):
    import ctypes as C

    from deepwmh_b200 import _lib
    lib = _lib.load()
    ws = _WS.setdefault("ws", torch.empty(_lib.DWMH_CT_WORKSPACE_BYTES, dtype=torch.uint8, device="cuda"))
    _lib.check(lib.dwmh_ct_normalize(0, C.c_void_p(v.data_ptr()), C.c_void_p(0), v.numel(), _lib.DWMH_NORM_CT2,
                                     c["percentile_00_5"], c["percentile_99_5"], 0.0, 1.0, None, C.c_void_p(ws.data_ptr()),
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream)))


def end_to_end(tmp, tta):
    plans = benchmark_plans(num_modalities=1, num_classes=3)
    st = plans["plans_per_stage"][0]
    full = dict(st, current_spacing=np.array([1.0, 0.8, 0.8]))
    low = dict(st, current_spacing=np.array([2.5, 2.0, 2.0]))
    plans = dict(plans, plans_per_stage={0: low, 1: full}, normalization_schemes={0: "CT"}, use_mask_for_norm={0: False},
                 dataset_properties={"intensityproperties": {0: CT}})
    root = os.path.join(tmp, "model")
    for model, trainer, M, seed in (("3d_fullres", "nnUNetTrainerV2", 1, 0), ("3d_lowres", "nnUNetTrainerV2", 1, 1),
                                    ("3d_cascade_fullres", "nnUNetTrainerV2CascadeFullRes", 3, 2)):
        tdir = os.path.join(root, "nnUNet", model, "Task003_Liver", "%s__nnUNetPlansv2.1" % trainer)
        os.makedirs(os.path.join(tdir, "all"))
        pickle.dump(plans, open(os.path.join(tdir, "plans.pkl"), "wb"))
        stage = {0: low} if model == "3d_lowres" else {1: full}
        net = O.build_benchmark_network(seed, dict(plans, plans_per_stage=stage, num_modalities=M))
        torch.save({"state_dict": net.state_dict()}, os.path.join(tdir, "all", "model_best.model"))
    os.environ["RESULTS_FOLDER"] = root
    shape = (300, 512, 512)                                                    # z, y, x
    rng = np.random.default_rng(0)
    z, y, x = np.ogrid[-1:1:300j, -1:1:512j, -1:1:512j]
    vol = np.full(shape, -1000, np.int16)
    vol[np.broadcast_to((y / 0.8) ** 2 + (x / 0.9) ** 2 < 1, shape)] = 40
    vol[np.broadcast_to(((y - 0.2) / 0.35) ** 2 + ((x + 0.3) / 0.3) ** 2 + (z / 0.7) ** 2 < 1, shape)] = 150
    vol = (vol + rng.integers(-25, 26, shape, dtype=np.int16)).astype(np.int16)
    indir = os.path.join(tmp, "in")
    os.makedirs(indir)
    nifti.write_nifti(os.path.join(indir, "ct_0000.nii.gz"), np.transpose(vol, (2, 1, 0)),
                      nifti.default_header(shape[::-1], spacing=(0.8, 0.8, 1.0)), dtype=np.int16)
    base = ["-i", indir, "-t", "Task003_Liver", "-f", "all", "-chk", "model_best", "--overwrite_existing"]
    if not tta:
        base.append("--disable_tta")
    small = os.path.join(tmp, "small")                                         # warm-up: CUDA context, modules, allocator
    os.makedirs(small)
    nifti.write_nifti(os.path.join(small, "ct_0000.nii.gz"), np.transpose(vol[:160, :200, :200], (2, 1, 0)),
                      nifti.default_header((200, 200, 160), spacing=(0.8, 0.8, 1.0)), dtype=np.int16)
    NP.main(["-i", small, "-o", os.path.join(tmp, "out_warm"), "-t", "Task003_Liver", "-f", "all", "-chk", "model_best",
             "-m", "3d_cascade_fullres", "--disable_tta"])
    for model in ("3d_fullres", "3d_lowres", "3d_cascade_fullres"):
        out = os.path.join(tmp, "out_%s" % model)
        torch.cuda.synchronize()
        t = time.perf_counter()
        NP.main(base + ["-o", out, "-m", model])
        torch.cuda.synchronize()
        secs = time.perf_counter() - t
        labels = np.transpose(nifti.read_nifti(os.path.join(out, "ct.nii.gz"))[0], (2, 1, 0))
        yield {"model": model, "case_shape_zyx": list(shape), "spacing_zyx": [1.0, 0.8, 0.8], "tta": bool(tta),
               "wall_s": round(secs, 2), "label_fractions": [round(float((labels == c).mean()), 4) for c in range(3)],
               "note": "file read to label file written; includes its own 3d_lowres pass" if model == "3d_cascade_fullres"
               else "file read to label file written", "status": "measured"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ct_r03.json"))
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--tta", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "ct_bench measures on the GPU; there is no CPU fallback"
    res = {"card": _card(), "kernels": kernels(args.iters), "end_to_end": []}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def save():
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    save()
    print(json.dumps(res["kernels"], indent=1), flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        for row in end_to_end(tmp, args.tta):                  # each row is saved as soon as it is measured
            res["end_to_end"].append(row)
            res["card_after"] = _card()
            save()
            print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
