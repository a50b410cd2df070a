"""Multi-GPU drivers for the path (SURVEY.md section 8e): one process per GPU, `torch.distributed`.

* cohort sharding  -- subjects are independent: subject i -> rank i mod world; no collective on
  the data path (only host-side gathers of names / timings).
* tile sharding    -- the tiles of ONE large volume are split into contiguous ranges per rank; every
  rank accumulates its tiles into its own full-size fp32 `agg`, then ONE collective (NCCL over NVLink
  on GPUs; gloo in the CPU tests) sums `agg` before finalize.  The weight buffer never crosses the
  link: it does not depend on the data, so every rank computes the complete one locally
  (`dwmh_weight_map`, bit-identical to a single-GPU run).  Collective variants (`reduce=`):
    "reduce"      ncclReduce to rank 0, which finalises (default: half the bytes of an all-reduce;
                  the result lives on rank 0, the rank that writes the NIfTI)
    "allreduce"   ncclAllReduce of agg, every rank finalises the whole volume (result on every rank)
    "allreduce2"  round 1's two all-reduces of agg and wgt (kept for the measured comparison)
* ensemble         -- k models resident on each rank (workspaces shared, `dwmh_create_like`), looped
  per subject; softmax mean and argmax on the device (a13).

Nothing in the reference corresponds to this file (it is single-GPU: deepwmh/main/predict.py:150).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

REDUCE_MODES = ("reduce", "allreduce", "allreduce2")


def shard_cohort(n_cases: int, rank: int, world: int) -> List[int]:
    """Static round-robin: equal-size volumes, so subject i goes to rank i mod world."""
    return list(range(rank, n_cases, world))


def shard_tiles(n_tiles: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous [begin, end) ranges in x-outer tile order (neighbouring tiles stay on one GPU, so the
    region each rank touches is a slab).  The first n_tiles % world ranks get one extra tile."""
    base, rem = divmod(n_tiles, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def _world(group=None) -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def reduce_aggregation(agg: torch.Tensor, wgt: Optional[torch.Tensor] = None, mode: str = "reduce", group=None) -> bool:
    """The one exchange step of the tile-sharded mode: sum agg [2,X,Y,Z] over ranks (and wgt only in the
    two-buffer variant).  Returns True on the ranks that hold the complete sum afterwards."""
    if mode not in REDUCE_MODES:
        raise ValueError("reduce mode %r (one of %s)" % (mode, ", ".join(REDUCE_MODES)))
    rank, world = _world(group)
    if world == 1:
        return True
    if mode == "reduce":
        dist.reduce(agg, dst=dist.get_global_rank(group, 0) if group is not None else 0, op=dist.ReduceOp.SUM, group=group)
        return rank == 0
    dist.all_reduce(agg, op=dist.ReduceOp.SUM, group=group)
    if mode == "allreduce2":
        if wgt is None:
            raise ValueError("allreduce2 needs the per-rank weight buffer")
        dist.all_reduce(wgt, op=dist.ReduceOp.SUM, group=group)
    return True


def allreduce_buffers(agg: torch.Tensor, wgt: torch.Tensor, group=None):
    """Round 1's exchange (two all-reduces); kept as the `allreduce2` variant."""
    reduce_aggregation(agg, wgt, "allreduce2", group)


def predict_volume_tile_sharded(trainer, data, do_mirroring=True, mirror_axes=(0, 1, 2), step_size=0.5,
                                use_gaussian=True, group=None, reduce: str = "reduce", timings: Optional[Dict] = None):
    """Tile-sharded predict_preprocessed_data_return_seg_and_softmax: every rank passes the same (c,x,y,z) array
    (numpy or a CUDA tensor) and the ranks holding the complete sum (rank 0, or all with an all-reduce) get
    (seg uint8 [x,y,z], softmax fp32 [C,x,y,z]) back as device tensors; the others get (None, None).
    timings (optional dict) receives device milliseconds of the stages {tiles, collective, finalize} (adds syncs)."""
    from .predictor import pad_nd_image
    net = trainer.network
    rank, world = _world(group)
    with torch.cuda.device(net.device):
        if isinstance(data, torch.Tensor) and data.is_cuda:
            vol = data.detach().to(device=net.device, dtype=torch.float32)
            diff = [max(p - s, 0) for p, s in zip(net.patch_size, vol.shape[1:])]
            pads = [(d // 2, d // 2 + d % 2) for d in diff]
            if any(diff):
                vol = torch.nn.functional.pad(vol, (pads[2][0], pads[2][1], pads[1][0], pads[1][1], pads[0][0], pads[0][1]))
            vol = vol.contiguous()
            sl = tuple(slice(b, vol.shape[i + 1] - a) for i, (b, a) in enumerate(pads))
        else:
            padded, slicer = pad_nd_image(np.asarray(data, dtype=np.float32), net.patch_size)
            vol = torch.from_numpy(np.ascontiguousarray(padded)).to(net.device)
            sl = tuple(slicer[1:])
        X, Y, Z = vol.shape[1:]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timings is not None else None
        agg = torch.zeros((net.num_classes, X, Y, Z), dtype=torch.float32, device=net.device)
        n_tiles = net.num_tiles((X, Y, Z), step_size)
        b, e = shard_tiles(n_tiles, rank, world)
        # use_gaussian must be decided on the GLOBAL tile count (the reference: num_tiles > 1)
        gauss = bool(use_gaussian) and n_tiles > 1
        # dwmh_predict_3d also accumulates the weights of this rank's tiles; only the two-buffer variant uses that partial
        # sum -- the one-collective modes overwrite wgt with the complete, locally computed map before finalize
        wgt = torch.zeros((X, Y, Z), dtype=torch.float32, device=net.device)
        if ev:
            ev[0].record()
        if e > b:
            net.accumulate_tiles(vol, agg, wgt, step_size, do_mirroring, mirror_axes, gauss, b, e)
        if ev:
            ev[1].record()
        complete = reduce_aggregation(agg, wgt if reduce == "allreduce2" else None, reduce, group)
        if ev:
            ev[2].record()
        seg = probs = None
        if complete:
            if reduce != "allreduce2":
                net.weight_map((X, Y, Z), step_size, gauss, out=wgt)
            seg, probs = net.finalize(agg, wgt)
            seg, probs = seg[sl], probs[(slice(None),) + sl]
        if ev:
            ev[3].record()
            torch.cuda.synchronize()
            timings.update(tiles_ms=ev[0].elapsed_time(ev[1]), collective_ms=ev[1].elapsed_time(ev[2]),
                           finalize_ms=ev[2].elapsed_time(ev[3]), collective_bytes=int(agg.numel() * 4 * (1.5 if reduce == "allreduce2" else 1.0)),
                           tiles=(b, e), n_tiles=n_tiles)
    return seg, probs


def ensemble_mean(softmaxes: Sequence[torch.Tensor]) -> torch.Tensor:
    """a13: np.mean(np.vstack(softmax), 0) over the k checkpoints (host / eager form, used by the CPU tests)."""
    acc = torch.zeros_like(softmaxes[0])
    for s in softmaxes:
        acc += s
    return acc / float(len(softmaxes))


def make_ensemble(plans: Dict, state_dicts: Sequence[Dict], device: int = 0, act_dtype: str = "fp16", max_batch: int = 32):
    """k resident models on one GPU: the first owns the activation workspaces, the others borrow them."""
    from .predictor import nnUNetTrainerV2
    trainers = []
    for sd in state_dicts:
        tr = nnUNetTrainerV2(plans, device=device, act_dtype=act_dtype, max_batch=max_batch,
                             share_workspace_with=trainers[0] if trainers else None)
        tr.load_checkpoint_ram({"state_dict": sd}, False)
        trainers.append(tr)
    return trainers


def predict_volume_ensemble(trainers: Sequence, vol: torch.Tensor, do_mirroring=True, mirror_axes=(0, 1, 2), step_size=0.5,
                            use_gaussian=True):
    """predict_cases' `for p in params` loop (a13) with every model resident: vol = normalised fp32 [X,Y,Z] (one modality) or
    [M,X,Y,Z] on the device (each extent >= patch) -> (seg uint8 [X,Y,Z], mean softmax fp32 [C,X,Y,Z]), all on the device: per
    model tiled prediction + finalize, running mean by dwmh_axpy (mean = sum_k softmax_k / k in model order), argmax by
    dwmh_argmax."""
    net0 = trainers[0].network
    k = len(trainers)
    with torch.cuda.device(net0.device):
        X, Y, Z = vol.shape[-3:]
        C = net0.num_classes
        mean = torch.zeros((C, X, Y, Z), dtype=torch.float32, device=net0.device)
        agg = torch.empty((C, X, Y, Z), dtype=torch.float32, device=net0.device)
        wgt = torch.empty((X, Y, Z), dtype=torch.float32, device=net0.device)
        for tr in trainers:
            agg.zero_(); wgt.zero_()
            tr.network.accumulate_tiles(vol, agg, wgt, step_size, do_mirroring, mirror_axes, use_gaussian)
            _, probs = tr.network.finalize(agg, wgt)
            net0.axpy_(mean, probs, 1.0 / k)
        seg = net0.argmax(mean)
    return seg, mean


def checkpoint_ensemble_refined_label(trainer, checkpoints: Sequence[dict], data, valid_mask=None, voxel_size=(1.0, 1.0, 1.0),
                                      do_mirroring: bool = False):
    """SURVEY 8f-3: stage-2 label refinement of deepwmh/pipeline/DCNN_multistage.py:317-394 without the NIfTI round trips.
    For each of the k epoch checkpoints: load it (`load_checkpoint_ram`), predict the volume (the reference disables TTA
    here, :334-336), keep the BACKGROUND probability x; accumulate y = 1 - m (1 - x) (`_parallel_softmax_masking`), average
    over k, label = field < 0.5, remove components below 3 mm^3 (`_parallel_ensembling`).
    data: preprocessed [1, X, Y, Z]; valid_mask: [X, Y, Z] array / tensor or None.
    -> (field fp32 [X, Y, Z], label uint8 [X, Y, Z]) as device tensors."""
    net = trainer.network
    k = len(checkpoints)
    if k == 0:
        raise ValueError("checkpoint_ensemble_refined_label: no checkpoints")
    acc = None
    m = None
    if valid_mask is not None:
        m = torch.as_tensor(np.ascontiguousarray(valid_mask) if isinstance(valid_mask, np.ndarray) else valid_mask)
        m = m.to(device=net.device, dtype=torch.float32).contiguous()
    for ck in checkpoints:
        trainer.load_checkpoint_ram(ck, False)
        _, softmax = trainer.predict_preprocessed_data_return_seg_and_softmax(
            data, do_mirroring=do_mirroring, mirror_axes=trainer.data_aug_params["mirror_axes"], use_sliding_window=True,
            step_size=0.5, use_gaussian=True, all_in_gpu=False, mixed_precision=True)
        bg = torch.as_tensor(softmax[0]).to(device=net.device, dtype=torch.float32).contiguous()
        if acc is None:
            acc = torch.zeros_like(bg)
        with torch.cuda.device(net.device):
            net.ensemble_masked_add_(acc, bg, m)
    with torch.cuda.device(net.device):
        label = net.ensemble_refine_(acc, k)
        label = net.remove_3mm_sparks(label, voxel_size)
    return acc, label
