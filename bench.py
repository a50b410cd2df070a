#!/usr/bin/env python
"""Headline benchmark of the hot path (BASELINE.json): volumes/sec of nnU-Net 3d_fullres sliding-window
inference with 8x mirror TTA + Gaussian aggregation on a synthetic 182x218x182 FLAIR volume,
Generic_UNet random-init, patch 128^3 (config[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1: cohort sharding, every rank runs K subjects, no collective on
the data path -> "scaling": "weak").  A step = one volume through z-score -> 12 tiles x 8 mirrors of
Generic_UNet -> overlap-add -> finalize.  `value` is timed with the raw volume already in HBM; `e2e` goes
through the C-ABI host-buffer call (dwmh_predict_volume_host) with pinned host memory, H2D + D2H inside.
`--impl reference` times the CPU oracle (the reference's PyTorch arithmetic, oracle/) on the host cores.
Prints ONE JSON line on rank 0.  `--dump-outputs DIR` also writes what the last timed step returned (see dump_outputs).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPE = (182, 218, 182)
N_TILES, N_MIRRORS = 12, 8
WORKLOAD = "synthetic 182x218x182 FLAIR, 3d_fullres Generic_UNet random-init (31.2M params), patch 128^3, step 0.5, 8x mirror TTA, Gaussian aggregation, z-score(nonzero mask)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": d["hbm_gbs"], "tensor_burst": d["bf16_tflops"], "tensor": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.limit"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons, pw, plim = [], None, set(), [], None
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            try:
                pw.append(float(r[2])); plim = float(r[7])
            except Exception:
                pass
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if mx and s > 0.3 * mx] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w": statistics.median(pw) if pw else None, "power_limit_w": plim}


# ------------------------------------------------------------------------------------------------
# CPU legs (the only places that execute oracle/): the reference arm and the own arm's cpu_baseline
# ------------------------------------------------------------------------------------------------
def _oracle_inputs(threads, seed=0):
    import torch
    import oracle as O
    torch.set_num_threads(threads)
    plans = O.benchmark_plans()
    net = O.build_benchmark_network(0, plans)
    return O, plans, net, O.synthetic_flair(SHAPE, seed=seed)


def cpu_whole_volume_no_tta(threads):
    """BASELINE config 1 as written: ONE whole 182x218x182 volume, z-score + sliding window WITHOUT mirroring (12 tile
    forwards), through the oracle's trainer surface.  Returns seconds."""
    O, plans, net, raw = _oracle_inputs(threads)
    tr = O.OracleTrainer(plans, net)
    t0 = time.perf_counter()
    data = raw.copy()
    data[0] = O.zscore_nnunet(raw[0], np.where(raw[0] != 0, 0, -1), True)
    tr.predict_preprocessed_data_return_seg_and_softmax(data, do_mirroring=False)
    return time.perf_counter() - t0


def run_reference(args):
    """Reference arm: the reference's arithmetic (oracle port: its engine is an un-vendored third-party package, nothing
    of it exists to run) on the host cores, SAME config as the own arm (8x TTA).  A step = one tile of the workload =
    8 mirrored forwards + softmax + Gaussian weighting + the host numpy overlap-add, driven through the oracle's own
    tiled predictor (generator form); every 12th step also pays the z-score of the next volume and the final
    divide + argmax.  value = (timed tiles / 12) / timed seconds."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count()
    O, plans, net, raw = _oracle_inputs(cores)

    def volume_steps(seed):
        r = O.synthetic_flair(SHAPE, seed=seed) if seed else raw
        t0 = time.perf_counter()
        data = r.copy()
        data[0] = O.zscore_nnunet(r[0], np.where(r[0] != 0, 0, -1), True)
        gen = O.iter_predict_3D_tiled(net, data, 0.5, True, (0, 1, 2), (128, 128, 128), True)
        carry = time.perf_counter() - t0               # z-score: charged to the volume's first tile
        while True:
            t0 = time.perf_counter()
            kind, *_ = next(gen)
            dt = time.perf_counter() - t0 + carry
            carry = 0.0
            if kind == "done":
                yield ("done", dt)
                return
            yield ("tile", dt)

    times, seed, gen = [], 0, None
    while len(times) < args.warmup + args.steps:
        if gen is None:
            gen = volume_steps(seed)
        kind, dt = next(gen)
        if kind == "done":                              # divide + argmax of a finished volume: charged to its last tile
            times[-1] += dt
            gen, seed = None, seed + 1
        else:
            times.append(dt)
    timed = times[args.warmup:]
    per_tile = sum(timed) / len(timed)
    vps = 1.0 / (per_tile * N_TILES)
    sample = ("each step = 1 of the 12 tiles of the workload (8 mirrored 128^3 forwards, softmax, x Gaussian/8, host numpy overlap-add; "
              "z-score / final divide + argmax charged to a volume's first / last tile), fp32 oracle port through its own tiled "
              "predictor, torch CPU %d threads; %d timed tiles = %.2f volumes" % (cores, len(timed), len(timed) / N_TILES))
    print(json.dumps({
        "impl": "reference", "metric": "volumes/sec", "value": vps, "unit": "volumes/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_tile * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD, "step_definition": "1/12 volume (one tile, 8 mirrors)"},
        "cpu_baseline": {"value": vps, "unit": "volumes/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": vps, "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def incumbent_cudnn(n_patches=4):
    """The incumbent Blackwell path (SURVEY 2.2): the same network in PyTorch through cuDNN with fp16 autocast (what
    nnU-Net's mixed_precision=True runs), on the same GPU.  A reported baseline like cpu_baseline; executes oracle/."""
    import torch
    import oracle as O
    net = O.build_benchmark_network(0, O.benchmark_plans()).cuda().eval()
    x = torch.randn(n_patches, 1, 128, 128, 128, device="cuda")
    torch.backends.cudnn.benchmark = True

    def f():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            return torch.softmax(net(x).float(), 1)
    f(); f(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        f()
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 3 / n_patches
    del net, x
    torch.cuda.empty_cache()
    return ms


# ------------------------------------------------------------------------------------------------
def conv_algorithmic_bytes(plans, raw32_max_edge=64):
    """Bytes every conv / transposed-conv launch of ONE tile-forward must move at least once: input activations
    (fp16; fp32 for the 1-channel input volume), output (fp16 raw, fp32 for layers whose output edge <= raw32_max_edge)
    and the layer's fp16 weights.  Returns (total bytes, number of launches)."""
    import numpy as np
    st = plans["plans_per_stage"][max(plans["plans_per_stage"].keys())]
    pools, kers = st["pool_op_kernel_sizes"], st["conv_kernel_sizes"]
    shape = np.array(st["patch_size"], dtype=np.int64)
    feats = [plans["base_num_features"]]
    for _ in pools:
        feats.append(min(int(round(feats[-1] * 2)), 320))
    total, launches, cin, shapes = 0, 0, plans["num_modalities"], []
    in_shape = shape.copy()

    def out_bytes(c, sp, last=False):
        return int(np.prod(sp)) * c * (4 if (max(sp) <= raw32_max_edge and not last) else 2)
    for d in range(len(pools) + 1):
        if d > 0:
            shape = shape // np.array(pools[d - 1])
        k = int(np.prod(kers[d]))
        total += int(np.prod(in_shape)) * cin * (4 if d == 0 else 2) + out_bytes(feats[d], shape) + cin * feats[d] * k * 2
        total += int(np.prod(shape)) * feats[d] * 2 + out_bytes(feats[d], shape) + feats[d] * feats[d] * k * 2
        launches += 2
        cin, in_shape = feats[d], shape.copy()
        shapes.append(shape.copy())
    for u in range(len(pools)):
        skip, sp = feats[-(2 + u)], shapes[-(2 + u)]
        k = int(np.prod(kers[-(u + 1)]))
        total += int(np.prod(in_shape)) * cin * 2 + int(np.prod(sp)) * skip * 2 + cin * skip * int(np.prod(pools[-(u + 1)])) * 2      # transposed conv
        total += int(np.prod(sp)) * 2 * skip * 2 + out_bytes(skip, sp) + 2 * skip * skip * k * 2
        total += int(np.prod(sp)) * skip * 2 + out_bytes(skip, sp, last=(u == len(pools) - 1)) + skip * skip * k * 2
        launches += 3
        cin, in_shape = skip, sp.copy()
    return total, launches


V2_SHAPE = (512, 512, 320)
DUMP_VOXELS = 1 << 22


def dump_outputs(out_dir, seg, probs):
    """The argmax [X,Y,Z] and softmax [2,X,Y,Z] of a timed step on a fixed, seeded sample of DUMP_VOXELS voxels (the same
    voxels in every run), as DIR/seg.npy [N] and DIR/softmax.npy [2,N] in float32: 48 MiB, so that two builds can be
    compared output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(seg.numel(), size=DUMP_VOXELS, replace=False))
    i = torch.from_numpy(idx).to(seg.device)
    np.save(os.path.join(out_dir, "seg.npy"), seg.reshape(-1)[i].float().cpu().numpy())
    np.save(os.path.join(out_dir, "softmax.npy"), probs.reshape(2, -1)[:, i].float().cpu().numpy())


def run_b200(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    import deepwmh_b200
    from deepwmh_b200 import parallel as PAR
    from deepwmh_b200 import workload as W      # synthetic volume + random-init weights (product side; oracle/ is only in the baseline legs)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pk = peaks()

    plans = deepwmh_b200.benchmark_plans()
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=local, act_dtype=args.dtype, max_batch=args.max_batch)
    tr.load_checkpoint_ram({"state_dict": W.random_init_state_dict(plans, 0)}, False)
    n = tr.network
    flops_fwd = W.forward_flops(plans)

    # per-rank subject (cohort sharding: rank r owns subjects r, r+world, ...)
    raws = [W.synthetic_flair(SHAPE, seed=rank + world * i)[0] for i in range(2)]
    raw_dev = [torch.from_numpy(r).to(dev) for r in raws]
    pinned = [torch.from_numpy(r).pin_memory() for r in raws]
    X, Y, Z = SHAPE
    V = X * Y * Z
    vol = torch.empty(SHAPE, dtype=torch.float32, device=dev)
    agg = torch.empty((2,) + SHAPE, dtype=torch.float32, device=dev)
    wgt = torch.empty(SHAPE, dtype=torch.float32, device=dev)
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > 126 MB L2
    sm_out = torch.empty((2,) + SHAPE, dtype=torch.float32).pin_memory()
    seg_out = torch.empty(SHAPE, dtype=torch.uint8).pin_memory()

    def step_device(i, net=None):
        net = net or n
        flush.zero_()
        vol.copy_(raw_dev[i % 2])                  # device-to-device: input resident in HBM
        net.normalize_(vol, None, 2, return_stats=False)
        agg.zero_(); wgt.zero_()
        net.accumulate_tiles(vol, agg, wgt, 0.5, True, (0, 1, 2), True)
        return net.finalize(agg, wgt)

    def step_e2e(i):
        flush.zero_()
        tr.predict_raw_volume_host(pinned[i % 2].numpy(), 2, True, (0, 1, 2), 0.5, True, sm_out.numpy(), seg_out.numpy())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, net=None):
        """-> (ms, kernel launches, what the last timed step returned)"""
        net = net or n
        for i in range(warmup):
            fn(i)
        barrier()
        k0, _ = net.counters()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            last = fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        k1, _ = net.counters()
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, k1 - k0, last

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev, launches, last = timed(step_device, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)     # before the next step overwrites agg, which holds the softmax
    del last
    ms_e2e, _, _ = timed(step_e2e, args.steps, 1)

    # roofline of the dominant kernel family (conv stack): device time of the conv stack, CUDA events
    # recorded by the library on the launching stream around the launches of one more volume
    n._lib.dwmh_set_stage_timing(n._ctx, 1)
    step_device(0); torch.cuda.synchronize()
    st = (C.c_float * 4)()
    n._lib.dwmh_get_stage_timing(n._ctx, st)
    kt = (C.c_double * 9)()
    n._lib.dwmh_get_kernel_timing(n._ctx, kt)
    n._lib.dwmh_set_stage_timing(n._ctx, 0)
    conv_ms, agg_ms, tc_ms, tc_tflop = float(st[0]), float(st[1]), float(st[2]), float(st[3])
    kinds = [n.layer_kernel_kind(i) for i in range(n.num_layers())]
    tc_launches_per_fwd = int(sum(kinds))

    # HBM-bound kernels timed alone
    def ev_time(fn, reps=5):
        fn(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    zs_ms = ev_time(lambda: (flush.zero_(), vol.copy_(raw_dev[0]), n.normalize_(vol, None, 2, return_stats=False))) - ev_time(lambda: (flush.zero_(), vol.copy_(raw_dev[0])))
    fin_ms = ev_time(lambda: (flush.zero_(), n.finalize(agg, wgt))) - ev_time(lambda: (flush.zero_(),))

    # ---- config 5: 5-model ensemble on the cohort (models resident, workspaces shared; softmax mean on the device) ----
    ens = None
    if args.ensemble > 1:
        trs = [tr] + [deepwmh_b200.nnUNetTrainerV2(plans, device=local, act_dtype=args.dtype, max_batch=args.max_batch, share_workspace_with=tr)
                      for _ in range(args.ensemble - 1)]
        for k, t_ in enumerate(trs[1:], 1):
            t_.load_checkpoint_ram({"state_dict": W.random_init_state_dict(plans, k)}, False)

        def step_ens(i):
            flush.zero_()
            vol.copy_(raw_dev[i % 2])
            n.normalize_(vol, None, 2, return_stats=False)
            return PAR.predict_volume_ensemble(trs, vol)
        es = max(1, min(args.steps, 3))
        ms_ens, _, _ = timed(step_ens, es, 1)
        ens = {"models": args.ensemble, "value": world * es / (ms_ens / 1e3), "unit": "volumes/s", "ms_per_volume": ms_ens / es,
               "forwards_per_volume": args.ensemble * N_TILES * N_MIRRORS, "steps": es,
               "note": "BASELINE config 5: every subject through %d resident random-init models (seeds 1234+k), 8x TTA each, softmax mean + argmax on the device; cohort sharded over %d GPU(s), no collective" % (args.ensemble, world)}
        for t_ in reversed(trs[1:]):
            t_.network.close()

    # ---- config 4: ONE 512x512x320 volume, tiles sharded over the ranks, one NCCL reduce of the fp32 aggregation buffer ----
    big = None
    if args.big_volume:
        raw2 = torch.from_numpy(W.synthetic_flair(V2_SHAPE, seed=0)[0]).to(dev)
        n.normalize_(raw2, None, 2, return_stats=False)
        data2 = raw2[None]
        tms = []
        ev_b = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
        res = None
        for it in range(1 + args.big_steps):
            tm = {}
            barrier()
            ev_b[0].record()
            res = PAR.predict_volume_tile_sharded(tr, data2, reduce=args.reduce, timings=None if it == 0 else tm)
            ev_b[1].record()
            barrier()
            if it > 0:
                tm["total_ms"] = ev_b[0].elapsed_time(ev_b[1])
                tms.append(tm)

        def over_ranks(key, op):
            v = sum(t[key] for t in tms) / len(tms)
            if world > 1:
                tt = torch.tensor([v], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=op)
                v = float(tt.item())
            return v

        def agg_max(key):
            return over_ranks(key, dist.ReduceOp.MAX)
        tot = sum(t["total_ms"] for t in tms) / len(tms)
        if world > 1:
            tt = torch.tensor([tot], device=dev, dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX); tot = float(tt.item())
        tiles_ms, coll_ms, fin2_ms = agg_max("tiles_ms"), agg_max("collective_ms"), agg_max("finalize_ms")
        tiles_min, coll_min = over_ranks("tiles_ms", dist.ReduceOp.MIN), over_ranks("collective_ms", dist.ReduceOp.MIN)
        big = {"shape": list(V2_SHAPE), "tiles": tms[0]["n_tiles"], "forwards": tms[0]["n_tiles"] * N_MIRRORS, "n_gpus": world,
               "s_per_volume": tot / 1e3, "volumes_per_s": 1e3 / tot, "tiles_ms_max_over_ranks": tiles_ms,
               "tiles_ms_min_over_ranks": tiles_min,
               "collective": args.reduce if world > 1 else "none (1 GPU)", "collective_ms_max_over_ranks": coll_ms,
               "collective_ms_min_over_ranks": coll_min,
               "collective_bytes": tms[0]["collective_bytes"] if world > 1 else 0,
               "collective_GBps": (tms[0]["collective_bytes"] / 1e9 / (coll_min / 1e3)) if (world > 1 and coll_min > 0) else None,
               "finalize_ms": fin2_ms, "steps": args.big_steps,
               "tflops": tms[0]["n_tiles"] * N_MIRRORS * flops_fwd / 1e12 / (tot / 1e3),
               "note": "BASELINE config 4: timed from the normalised volume in HBM to seg + softmax on rank 0 (zeroing of the buffers, this rank's tiles, "
                       "the collective, weight map + finalize).  collective_ms is measured per rank from the end of its own tiles: the MAX over ranks contains the wait "
                       "for the slowest rank (tile-time skew between GPUs), the MIN is the rank that arrived last, i.e. the transfer itself; GB/s uses the MIN"}
        if world > 1:
            # agreement with the single-GPU result of the same volume (rank 0 computes it once, untimed)
            if rank == 0:
                seg_s, p1_s = res[0].clone(), res[1][1].clone()
                agg1 = torch.zeros((2,) + V2_SHAPE, dtype=torch.float32, device=dev)
                wgt1 = torch.zeros(V2_SHAPE, dtype=torch.float32, device=dev)
                n.accumulate_tiles(raw2, agg1, wgt1, 0.5, True, (0, 1, 2), True)
                seg1, p1 = n.finalize(agg1, wgt1)
                big["vs_single_gpu"] = {"argmax_agree": float((seg1 == seg_s).double().mean().item()),
                                        "softmax_max_abs": float((p1[1] - p1_s).abs().max().item()),
                                        "note": "fp32 summation order of the overlap-add differs across shard counts (partial buffers are summed by the collective)"}
                del agg1, wgt1, seg1, p1, seg_s, p1_s
            barrier()
        del res
        del raw2, data2

    # ---- bf16 operands / storage (north_star's nominal dtype): speed beside the fp16 default; it fails the argmax gate ----
    alt = None
    if args.alt_dtype and rank == 0 and world == 1:
        other = "bf16" if args.dtype == "fp16" else "fp16"
        n_alt = None
        try:
            tr_alt = deepwmh_b200.nnUNetTrainerV2(plans, device=local, act_dtype=other, max_batch=args.max_batch)
            tr_alt.load_checkpoint_ram({"state_dict": W.random_init_state_dict(plans, 0)}, False)
            n_alt = tr_alt.network
            s_ref, _ = step_device(0)
            s_ref = s_ref.clone()
            ms_alt, _, _ = timed(lambda i: step_device(i, n_alt), 3, 2, n_alt)
            s_alt, _ = step_device(0, n_alt)
            alt = {"dtype": other, "value": 3 / (ms_alt / 1e3), "unit": "volumes/s", "ms_per_step": ms_alt / 3,
                   "argmax_agreement_with_%s_run" % args.dtype: float((s_alt == s_ref).float().mean().item())}
        except Exception as e:      # memory pressure on a shared box must not take the headline down
            alt = {"dtype": other, "error": str(e)[:200]}
        finally:
            if n_alt is not None:
                n_alt.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    vps = world * args.steps / (ms_dev / 1e3)
    vps_e2e = world * args.steps / (ms_e2e / 1e3)
    tflop_vol = flops_fwd * N_TILES * N_MIRRORS / 1e12
    n_batches = -(-N_TILES * N_MIRRORS // args.max_batch)
    tc_launches = tc_launches_per_fwd * n_batches
    achieved = tc_tflop / (tc_ms / 1e3)            # dominant kernel: conv3_tc_kernel (all tcgen05 conv / tconv launches)
    cores = os.cpu_count()
    cpu = None
    if args.cpu_baseline and world == 1:           # N = 1 only: bounded sample of ~10-30 s
        t_cpu = cpu_whole_volume_no_tta(cores)
        cpu = {"value": 1.0 / (t_cpu * N_MIRRORS), "unit": "volumes/s", "cores": cores, "kind": "port",
               "no_tta_volumes_per_s": 1.0 / t_cpu,
               "sample": "ONE whole 182x218x182 volume WITHOUT mirroring (BASELINE config 1: z-score + 12 tile forwards + host aggregation + argmax) through "
                         "OracleTrainer.predict_preprocessed_data_return_seg_and_softmax, fp32 oracle port, torch CPU %d threads: %.1f s; "
                         "value = 1 / (8 x that) for the 8x-TTA workload of this line" % (cores, t_cpu)}
    inc = None
    if args.incumbent and world == 1:
        try:
            ms_patch = incumbent_cudnn()
            inc = {"ms_per_patch": ms_patch, "volumes_per_s_equivalent": 1e3 / (ms_patch * N_TILES * N_MIRRORS),
                   "what": "the oracle's PyTorch Generic_UNet on this GPU through cuDNN, fp16 autocast (nnU-Net mixed_precision=True), 4 patches of 128^3 per call, forwards only"}
        except Exception as e:
            inc = {"error": str(e)[:200]}
    # DRAM traffic per conv3_tc_kernel launch cannot be measured inside a timed run: it is the committed ncu pass of the same
    # binary and command (tools/dram_traffic.py -> profiles/dram_traffic_r02b.json, else the earlier files)
    ab, nl = conv_algorithmic_bytes(plans)
    alg_bytes = ab * args.max_batch / nl          # mean over the conv launches of one max_batch-forward batch
    traffic, traffic_src = None, None
    for name in ("dram_traffic_r02b.json", "dram_traffic_r02.json", "dram_traffic_r01.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.isfile(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj["tc_dram_bytes_per_launch"]
                traffic_src = "COMMITTED CONSTANT, not measured in this run: profiles/%s (ncu dram__bytes_read.sum + dram__bytes_write.sum, mean over the %d conv3_tc_kernel launches of one 32-forward batch)" % (name, tj["tc_launches"])
                break
            except Exception:
                traffic = None
    P = 128 ** 3
    agg_bytes = N_TILES * P * (N_MIRRORS * 8 + 4 + 24.0)       # per tile voxel: M x 2 probabilities read, Gaussian read, agg[2] + wgt read-modify-write
    out = {
        "metric": "volumes/sec", "value": vps, "unit": "volumes/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16" if args.dtype == "fp16" else "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "forwards_per_volume": N_TILES * N_MIRRORS, "tflop_per_volume": tflop_vol,
                   "accumulate": "f32", "instance_norm_stats": "per-CTA Welford partials (f32) combined in a fixed order in f64: deterministic", "batch_forwards": args.max_batch,
                   "parallelism": "cohort x%d (one subject stream per GPU, no collective)" % world,
                   "l2": "192 MiB flush buffer written between steps; per-batch activation working set (~7 GB) >> 126 MB L2",
                   "tcgen05_layers": int(sum(kinds)), "direct_layers": int(len(kinds) - sum(kinds)),
                   "dtype_note": "fp16 operands/storage, the reference's own autocast type; bf16 (BASELINE config 2's nominal type) runs at the same rate but fails the 99.9 % argmax gate on random-init weights (profiles/precision_probe_r01.txt); see alt_dtype"},
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": achieved / pk["tensor"],
                     "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": alg_bytes, "kernel": "conv3_tc_kernel (tcgen05 implicit-GEMM conv3d / strided conv / transposed conv)",
                     "launches_per_volume": tc_launches, "avg_launch_ms": tc_ms / max(tc_launches, 1), "tflop_per_volume_in_kernel": tc_tflop,
                     "kernel_ms_per_volume": tc_ms, "kernel_share_of_step": tc_ms / (ms_dev / args.steps),
                     "conv_stack_ms_per_volume": conv_ms, "conv_stack_tflops": tflop_vol / (conv_ms / 1e3),
                     "whole_step_tflops": tflop_vol / (ms_dev / args.steps / 1e3), "whole_step_frac": tflop_vol / (ms_dev / args.steps / 1e3) / pk["tensor"],
                     "aggregate_ms_per_volume": agg_ms,
                     "peak_source": pk["src"] + ": sustained bf16 cuBLAS (the kernel runs inside a long step); burst %.1f" % pk["tensor_burst"]},
        "hbm_kernels": {"zscore": {"ms": zs_ms, "GBps": 12.0 * V / 1e9 / (zs_ms / 1e3), "frac_of_measured_hbm": 12.0 * V / 1e9 / (zs_ms / 1e3) / pk["hbm"]},
                        "finalize": {"ms": fin_ms, "GBps": 21.0 * V / 1e9 / (fin_ms / 1e3), "frac_of_measured_hbm": 21.0 * V / 1e9 / (fin_ms / 1e3) / pk["hbm"]},
                        "instnorm_lrelu": {"ms_per_volume": kt[3], "launches_per_volume": kt[5], "GBps": kt[4] / 1e9 / (kt[3] / 1e3) if kt[3] > 0 else None,
                                           "frac_of_measured_hbm": (kt[4] / 1e9 / (kt[3] / 1e3) / pk["hbm"]) if kt[3] > 0 else None},
                        "head_softmax": {"ms_per_volume": kt[6], "launches_per_volume": kt[8], "GBps": kt[7] / 1e9 / (kt[6] / 1e3) if kt[6] > 0 else None,
                                         "frac_of_measured_hbm": (kt[7] / 1e9 / (kt[6] / 1e3) / pk["hbm"]) if kt[6] > 0 else None},
                        "aggregate_tile": {"ms_per_volume": agg_ms, "launches_per_volume": N_TILES, "GBps": agg_bytes / 1e9 / (agg_ms / 1e3) if agg_ms > 0 else None,
                                           "frac_of_measured_hbm": (agg_bytes / 1e9 / (agg_ms / 1e3) / pk["hbm"]) if agg_ms > 0 else None},
                        "note": "zscore / finalize: timed alone with an L2 flush before each launch (87 / 152 MB algorithmic); the others: CUDA events around every launch of one volume, algorithmic bytes"},
        "cpu_baseline": cpu,
        "incumbent_cudnn": inc,
        "e2e": {"value": vps_e2e, "unit": "volumes/s", "h2d_bytes_per_step": 4 * V, "d2h_bytes_per_step": 9 * V,
                "ms_per_step": ms_e2e / args.steps, "api": "dwmh_predict_volume_host (C ABI, pinned host buffers)"},
        "ensemble5": ens,
        "tile_sharded": big,
        "alt_dtype": alt,
        "gpu_launches": int(launches), "clocks": clocks,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--max-batch", type=int, default=32)
    ap.add_argument("--cpu-baseline", type=int, default=1, help="N = 1: time one whole no-TTA volume with the CPU oracle (about 15 s; 0 = skip)")
    ap.add_argument("--incumbent", type=int, default=1, help="N = 1: time the PyTorch/cuDNN fp16-autocast forward of the same network (0 = skip)")
    ap.add_argument("--ensemble", type=int, default=5, help="models of the ensemble block (BASELINE config 5); 0/1 = skip")
    ap.add_argument("--big-volume", type=int, default=1, help="512x512x320 tile-sharded block (BASELINE config 4); 0 = skip")
    ap.add_argument("--big-steps", type=int, default=2)
    ap.add_argument("--reduce", default="reduce", choices=["reduce", "allreduce", "allreduce2"], help="collective of the tile-sharded block")
    ap.add_argument("--alt-dtype", type=int, default=1, help="N = 1: also time the other operand type (bf16 beside fp16)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's seg / softmax to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the b200 path's outputs; the reference arm times single tiles")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.gpus > 1 and "RANK" not in os.environ:
            # convenience: self-launch one rank per GPU
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
                   "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
            sys.exit(subprocess.call(cmd))
        run_b200(args)


if __name__ == "__main__":
    main()
