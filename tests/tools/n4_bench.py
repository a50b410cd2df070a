"""Device N4 bias-field correction (dwmh_n4) at BASELINE.json's 182x218x182 volume with DeepWMH's schedule (-s 2,
50x50x50x50): device time per call (CUDA events, median over repeated calls after warm-up), kernels per call (counted
with torch.profiler and against the schedule's count), one timed run of the fp64 numpy restatement (oracle/n4_oracle.py)
and the device result against it, with the card's name and power limit read in the same run.  Prints one JSON line.
The shrunk working set (two fp32 arrays of 91 x 109 x 91 = 3.6 MB each plus lattices and tables) stays in the 126 MB L2
across the 200 iterations of a call, so no L2 flush is done between calls: the first iteration of a call reads the
full-resolution volume from HBM once, everything after it runs out of L2.
usage: python tests/tools/n4_bench.py [--repeats N] [--out FILE]"""
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
from deepwmh_b200.n4 import n4_bias_field_correction  # noqa: E402
from oracle import n4_oracle as N  # noqa: E402

SHAPE = (182, 218, 182)
SCHEDULE = (50, 50, 50, 50)


def expected_kernels(schedule):
    """shrink + log; per level: [refine], tables, three omega kernels; 6 per iteration; output."""
    return 1 + sum(4 + (level > 0) for level in range(len(schedule))) + 6 * sum(schedule) + 1


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    name, plim, smax = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(plim), "sm_max_mhz": float(smax), "torch_name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=30)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    img, _, _ = N.phantom(SHAPE, seed=0)
    t = torch.from_numpy(img).cuda()
    run = lambda: n4_bias_field_correction(t, 2, SCHEDULE, return_log_field=True)
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    ms = []
    for _ in range(args.repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    t0 = time.time()
    for _ in range(5):
        run()
    torch.cuda.synchronize()
    wall_ms = (time.time() - t0) / 5 * 1e3

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.name.find("n4_") >= 0]
    per_kernel = {}
    for e in kern:
        d = per_kernel.setdefault(e.name[e.name.find("n4_"):].split("(")[0], [0, 0.0])
        d[0] += 1
        d[1] += getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
    out_d, field_d = [x.cpu().numpy() for x in run()]

    t0 = time.time()
    ref_out, ref_field = N.n4(img, 2, SCHEDULE, return_log_field=True)
    cpu_s = time.time() - t0
    v = img > 0
    res = {
        "workload": "N4 %dx%dx%d, shrink 2, iterations %s" % (SHAPE + ("x".join(map(str, SCHEDULE)),)),
        "device_ms_median": round(float(np.median(ms)), 3), "device_ms_min": round(float(np.min(ms)), 3),
        "device_ms_max": round(float(np.max(ms)), 3), "repeats": args.repeats,
        "wall_ms_per_call_with_sync": round(wall_ms, 3),
        "timing": "CUDA events around one call after 3 warm-up calls; the shrunk working set (2 x 3.6 MB fp32 + tables) is "
                  "L2-resident across the call's iterations, no L2 flush between calls",
        "kernels_per_call_profiled": len(kern), "kernels_per_call_expected": expected_kernels(SCHEDULE),
        "host_launches_per_call": {"kernels": expected_kernels(SCHEDULE) - 6 * sum(SCHEDULE), "graph_launches": sum(SCHEDULE),
                                   "graphs_instantiated": sum(1 for n in SCHEDULE if n > 0)},
        "kernel_us_per_call": {k: {"launches": c, "us": round(us, 1)} for k, (c, us) in sorted(per_kernel.items())},
        "oracle_cpu_s": round(cpu_s, 2), "oracle_cores": os.cpu_count(),
        "log_field_max_abs_diff": float(np.abs(field_d.astype(np.float64) - ref_field).max()),
        "corrected_max_rel_diff_valid": float((np.abs(out_d.astype(np.float64) - ref_out)[v] / np.abs(ref_out[v])).max()),
        "card": card(),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
