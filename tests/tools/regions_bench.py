"""Cost of region-based (sigmoid-head) models on one B200: one JSON line, also written to --out.

On the 128^3 benchmark plan with four modalities (random-init weights):
  * fwd32_ms / head_ms   a batch of 32 forwards (dwmh_forward_patches, CUDA events, median of --reps) and the head kernel's
                         device time in it (torch.profiler), for 3 sigmoid outputs next to 4 softmax classes;
  * region_labels        dwmh_region_labels device time (CUDA events over --label-reps launches) and the GB/s of its
                         4 R + 1 bytes per voxel, at 182 x 218 x 182 and 512 x 512 x 320, next to dwmh_argmax over 4 classes;
  * volume_ms            one 182 x 218 x 182 volume with 8x mirroring through predict_3D on device tensors with
                         regions_class_order (finalize + region labels included), median.
The card name and power limit are read in the same run (nvidia-smi query).

    python tests/tools/regions_bench.py [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import deepwmh_b200  # noqa: E402
import oracle as O  # noqa: E402
import regions_oracle as RO  # noqa: E402
from multimodal_bench import card  # noqa: E402

M = 4


def head_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    t = 0.0
    for e in prof.events():
        if "head_softmax" in e.name:
            t += (e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total) / 1000.0
    return t


def events_ms(fn, reps):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def trainer(sigmoid):
    if sigmoid:
        plans = deepwmh_b200.benchmark_plans(num_modalities=M, num_classes=4)
        net = RO.build_region_network(plans, 0, 3)
        tr = deepwmh_b200.nnUNetTrainerV2BraTSRegions(plans, device=0, max_batch=32)
    else:
        plans = deepwmh_b200.benchmark_plans(num_modalities=M, num_classes=4)
        net = O.build_benchmark_network(0, plans)
        tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=32)
    tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
    return tr


def forward_row(tr, reps):
    dev = tr.network
    x = torch.randn((32, M, 128, 128, 128), device="cuda")
    dev.forward_patches(x)
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); dev.forward_patches(x); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return {"nonlin": dev.inference_nonlin, "outputs": dev.num_classes, "fwd32_ms": round(float(np.median(ts)), 3),
            "head_ms": round(head_ms(lambda: dev.forward_patches(x)), 3)}


def label_rows(dev, reps):
    rows = []
    for shape in ((182, 218, 182), (512, 512, 320)):
        V = int(np.prod(shape))
        p = torch.rand((3,) + shape, device="cuda")
        ms = events_ms(lambda: dev.region_labels(p, (1, 2, 3)), reps)
        p4 = torch.rand((4,) + shape, device="cuda")
        ms_arg = events_ms(lambda: dev.argmax(p4), reps)
        rows.append({"shape": list(shape), "region_labels_ms": round(ms, 4), "region_labels_GBps": round((4 * 3 + 1) * V / ms / 1e6, 1),
                     "argmax4_ms": round(ms_arg, 4), "argmax4_GBps": round((4 * 4 + 1) * V / ms_arg / 1e6, 1)})
        del p, p4
    return rows


def volume_ms(tr, reps):
    dev = tr.network
    vol = torch.from_numpy(np.stack([O.synthetic_flair((182, 218, 182), seed=m)[0] for m in range(M)])).cuda()
    for m in range(M):
        dev.normalize_(vol[m], None, 2, return_stats=False)

    def run():
        return dev.predict_3D(vol, True, use_sliding_window=True, step_size=0.5, use_gaussian=True,
                              regions_class_order=tr.regions_class_order, return_device_tensors=True)
    run()
    vs = []
    for _ in range(reps):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        run()
        torch.cuda.synchronize()
        vs.append((time.perf_counter() - t0) * 1e3)
    return round(float(np.median(vs)), 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--label-reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("regions_bench needs a CUDA device")
    name, pl = card()
    sig = trainer(True)
    rows = [forward_row(sig, args.reps)]
    soft = trainer(False)
    rows.append(forward_row(soft, args.reps))
    soft.network.close()
    labels = label_rows(sig.network, args.label_reps)
    vms = volume_ms(sig, max(2, args.reps // 2))
    sig.network.close()
    line = json.dumps({"tool": "regions_bench", "gpu": name, "power_limit": pl, "plan": "128^3, 5 poolings, base 32, fp16, 4 modalities",
                       "forward": rows, "labels": labels,
                       "volume": {"shape": [182, 218, 182], "tta": 8, "regions_class_order": [1, 2, 3], "predict_3D_ms": vms}})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
