"""nnU-Net postprocessing.json on the device (dwmh_keep_largest_components, DESIGN §11): for the empty json, [1] and
[[1, 2], 1, 2] on seeded three-class label maps of 182x218x182 and 512x512x320, the device time of one whole json (CUDA
events, median over repeated calls after warm-up; the map is restored from a copy before each call, outside the timed
region), the launches per entry (the context's launch counter) with per-kernel times from torch.profiler, the host time
of the scipy restatement (tests/postprocessing_oracle.py) and whether the device result equals it bit for bit, with the
card's name and power limit read in the same run.  Prints one JSON line.
Working set per entry: the uint8 map plus two int32 arrays (labels, component sizes) of the map's voxel count, i.e. 65 MB
at 182x218x182, which fits in the 126 MB L2 (no flush between calls), and 755 MB at 512x512x320, which does not.
usage: python tests/tools/postprocessing_bench.py [--repeats N] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import deepwmh_b200  # noqa: E402
from deepwmh_b200 import postprocessing as PP  # noqa: E402
import postprocessing_oracle as PO  # noqa: E402
from conftest import small_plans  # noqa: E402

SHAPES = [(182, 218, 182), (512, 512, 320)]
JSONS = {"empty": [], "[1]": [1], "[[1,2],1,2]": [(1, 2), 1, 2]}
VPV = 1.0


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    name, plim, smax = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(plim), "sm_max_mhz": float(smax), "torch_name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    tr = deepwmh_b200.nnUNetTrainerV2(small_plans(), device=0, max_batch=1)
    net = tr.network
    rows = []
    for shape in SHAPES:
        seg = PO.label_map(shape, seed=0, sigma=2.0, scatter=0.005)
        src = torch.from_numpy(seg).cuda()
        d = torch.empty_like(src)
        classes = {c: int((seg == c).sum()) for c in range(3)}
        for tag, fwc in JSONS.items():
            run = lambda: PP.remove_all_but_the_largest_connected_component(net, d, fwc, VPV)
            for _ in range(3):
                d.copy_(src); run()
            torch.cuda.synchronize()
            ms = []
            for _ in range(args.repeats):
                d.copy_(src)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); run(); b.record()
                torch.cuda.synchronize()
                ms.append(a.elapsed_time(b))
            from torch.profiler import ProfilerActivity, profile
            d.copy_(src); torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run()
                torch.cuda.synchronize()
            kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "ccl_" in e.name]
            per_kernel = {}
            for e in kern:
                k = per_kernel.setdefault(e.name[e.name.find("ccl_"):].split("(")[0].split("<")[0], [0, 0.0])
                k[0] += 1
                k[1] += getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
            got = d.cpu().numpy()
            d.copy_(src)
            n0 = net.counters()[0]
            run()
            launches = net.counters()[0] - n0
            t0 = time.time()
            ref = PO.remove_all_but_the_largest_connected_component(seg, fwc, VPV)
            host_s = time.time() - t0
            rows.append({
                "shape": "x".join(map(str, shape)), "json": tag, "entries": len(fwc),
                "device_ms_median": round(float(np.median(ms)), 4), "device_ms_min": round(float(np.min(ms)), 4),
                "device_ms_max": round(float(np.max(ms)), 4),
                "launches_per_entry": (launches / len(fwc)) if fwc else 0, "kernels_profiled": len(kern),
                "kernel_us": {k: {"launches": c, "us": round(us, 1)} for k, (c, us) in sorted(per_kernel.items())},
                "oracle_host_s": round(host_s, 3), "bit_equal": bool(np.array_equal(got, ref)),
                "voxels_removed": int((got != seg).sum()), "voxels_per_class": classes,
            })
        del src, d
        torch.cuda.empty_cache()
    net.close()
    res = {
        "workload": "postprocessing.json on seeded three-class uint8 label maps (smooth blobs + 0.5 % scattered voxels), "
                    "volume_per_voxel 1.0",
        "timing": "CUDA events around one whole json after 3 warm-up calls, median of %d; the map is restored from a device "
                  "copy before each call, outside the timed region; no L2 flush (182x218x182: 65 MB working set, L2-resident; "
                  "512x512x320: 755 MB, exceeds the 126 MB L2)" % args.repeats,
        "oracle": "tests/postprocessing_oracle.py (scipy.ndimage.label + bincount) on %d host cores" % os.cpu_count(),
        "rows": rows, "card": card(),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
