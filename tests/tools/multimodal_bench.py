"""Cost of extra modalities and classes on one B200: one JSON line.

For M in {1, 2, 4} modalities and C in {2, 3, 4} classes on the 128^3 benchmark plan (random-init weights):
  * fwd32_ms        ms per batch of 32 forwards (dwmh_forward_patches, CUDA events, median of --reps)
  * first_conv_ms   device time of the first conv's kernel in that batch (torch.profiler)
  * head_ms         device time of the head kernel in that batch (torch.profiler)
  * volume_ms       ms per 182 x 218 x 182 volume with 8x mirroring (dwmh_predict_volume_host incl. H2D / D2H, median)
The card name and power limit are read in the same run (nvidia-smi query).

    python tests/tools/multimodal_bench.py [--reps 5] [--out FILE]
"""
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

import deepwmh_b200  # noqa: E402
import oracle as O  # noqa: E402


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], text=True)
        name, pl = [s.strip() for s in out.strip().splitlines()[0].split(",")]
        return name, pl
    except Exception as e:          # the numbers stay usable without it
        return torch.cuda.get_device_name(0), "unknown (%s)" % type(e).__name__


def kernel_ms(fn):
    """Device ms of the first-conv and head kernels of one call of fn (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    first = head = 0.0
    for e in prof.events():
        name = e.name
        t = e.device_time_total / 1000.0 if hasattr(e, "device_time_total") else e.cuda_time_total / 1000.0
        if "conv_first" in name or ("conv3_tc_kernel" in name and _is_first(name)):
            first += t
        elif "head_softmax" in name:
            head += t
    return first, head


def _is_first(name):
    # demangled: conv3_tc_kernel<T, KSTEPS, SMALL_CB, TCONV, DUAL, XFORM, FIRST>
    args = name.split("<", 1)[1].split(">", 1)[0].split(",")
    return len(args) >= 7 and args[6].strip() == "true"


def run(M, C, reps, vol_shape=(182, 218, 182)):
    plans = deepwmh_b200.benchmark_plans(num_modalities=M, num_classes=C)
    net = O.build_benchmark_network(0, plans)
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=32)
    tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
    dev = tr.network
    x = torch.randn((32, M, 128, 128, 128), device="cuda")
    dev.forward_patches(x)
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); dev.forward_patches(x); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    first, head = kernel_ms(lambda: dev.forward_patches(x))
    vol = O.synthetic_flair(vol_shape, seed=0)[0].astype(np.float32)
    v = np.ascontiguousarray(np.stack([vol * (1.0 + 0.25 * m) for m in range(M)]) if M > 1 else vol)
    tr.predict_raw_volume_host(v)
    vs = []
    for _ in range(max(2, reps // 2)):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        tr.predict_raw_volume_host(v)
        vs.append((time.perf_counter() - t0) * 1e3)
    dev.close()
    return {"M": M, "C": C, "fwd32_ms": round(float(np.median(ts)), 3), "first_conv_ms": round(first, 3),
            "head_ms": round(head, 3), "volume_ms": round(float(np.median(vs)), 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, pl = card()
    rows = [run(M, C, args.reps) for M in (1, 2, 4) for C in (2, 3, 4)]
    line = json.dumps({"tool": "multimodal_bench", "gpu": name, "power_limit": pl, "plan": "128^3, 5 poolings, base 32, fp16",
                       "volume": [182, 218, 182], "tta": 8, "rows": rows})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
