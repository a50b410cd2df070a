"""The tiled prediction (`dwmh_predict_3d` + `dwmh_finalize`) against a float64 aggregation of the device's own forwards.

The host rebuilds the device's call: the tile origins of `compute_steps_for_sliding_window`, tiles in x / y / z-inner
order, the mirrors m = 0..7 the device runs (bit 1 flips z, 2 flips y, 4 flips x; only those whose axes are enabled), and
the same batches (`max_batch // M` tiles of M forwards each, the last one shorter, counted from the first tile of the
range).  Each tile is cut out of the volume, flipped, and run through `forward_patches` as one call per device batch:
the batch size decides the z-block grouping of the conv kernels, and with equal batches the patch-mode forward (a
contiguous patch) and the tile-mode forward (the first conv's fetcher reading tile origin and flip from the volume) are
expected to be bit-identical.  Unflip, mirror average, importance map (scipy's, as installed), overlap-add and division
then run in float64.  What is left between the two is the device's fp32 overlap-add of at most 8 tiles.

So the check sees the fetcher's halo (zero padding at the patch edge, not the neighbouring tile's voxels), the unflip of
every mirror and every tile origin -- errors the end-to-end oracle test hides under the Gaussian map's small border
weights and the mirror average.  Two perturbed references, one mirror's z-unflip skipped and one tile origin moved by a
voxel, must each differ from the device result by 100 times the tolerance, which shows that both would be caught.
"""
import itertools

import numpy as np
import pytest
import torch

import oracle as O
from conftest import small_plans

SOFTMAX_TOL = 4e-6          # fp32 overlap-add of at most 8 tiles and one division
SEG_MARGIN = 1e-5           # the label must agree wherever the reference's |p1 - p0| exceeds this
WGT_RTOL = 1e-6
SENS_MIN = 100.0


def mirror_list(do_mirroring, mirror_axes):
    if not do_mirroring:
        return [0]
    need = {1: 2, 2: 1, 4: 0}          # mirror bit -> volume axis it flips
    return [m for m in range(8) if all(a in mirror_axes for b, a in need.items() if m & b)]


def flip_dims(m, lead):
    """Axes of a [..., x, y, z] tensor with `lead` leading dims that mirror m flips."""
    return [lead + a for b, a in ((1, 2), (2, 1), (4, 0)) if m & b]


class Reconstruction:
    """The device's tiled call restated on the host: forwards through `forward_patches`, everything else in float64."""

    def __init__(self, nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, ranges=((0, -1),)):
        ps = tuple(nw.patch_size)
        steps = O.compute_steps_for_sliding_window(ps, vol.shape, step_size)
        self.ps, self.shape = ps, tuple(vol.shape)
        self.origins = [(x, y, z) for x in steps[0] for y in steps[1] for z in steps[2]]
        self.mirrors = mirror_list(do_mirroring, mirror_axes)
        M = len(self.mirrors)
        per_batch = max(1, max_batch // M)
        if use_gaussian and len(self.origins) > 1:
            self.g = torch.from_numpy(O.get_gaussian(ps)).to(vol.device, torch.float64)
        else:
            self.g = torch.ones(ps, dtype=torch.float64, device=vol.device)
        self.probs = {}                   # tile index -> the M mirrored forwards as [M, 2, *patch] fp64, still flipped
        for b, e in ranges:
            e = len(self.origins) if e < 0 else e
            for t0 in range(b, e, per_batch):
                tiles = range(t0, min(t0 + per_batch, e))
                patches = torch.stack([self.tile(vol, t).flip(flip_dims(m, 0)) for t in tiles for m in self.mirrors])
                p = nw.forward_patches(patches[:, None].contiguous()).double()
                for k, t in enumerate(tiles):
                    self.probs.setdefault(t, []).append(p[k * M:(k + 1) * M])

    def tile(self, vol, t, origin=None):
        o = self.origins[t] if origin is None else origin
        return vol[o[0]:o[0] + self.ps[0], o[1]:o[1] + self.ps[1], o[2]:o[2] + self.ps[2]]

    def aggregate(self, skip_z_unflip=None, moved=None):
        """(softmax, weight sum) in float64.  skip_z_unflip = (tile, mirror index): leave that forward's z axis flipped;
        moved = (tile, origin): add that tile at another origin."""
        dev = self.g.device
        agg = torch.zeros((2,) + self.shape, dtype=torch.float64, device=dev)
        wgt = torch.zeros(self.shape, dtype=torch.float64, device=dev)
        M = len(self.mirrors)
        for t, parts in self.probs.items():
            for p in parts:                       # one entry per call that covered the tile
                r = torch.zeros((2,) + self.ps, dtype=torch.float64, device=dev)
                for j, m in enumerate(self.mirrors):
                    dims = flip_dims(m, 1)
                    if skip_z_unflip == (t, j):
                        dims = [d for d in dims if d != 3]
                    r += (p[j].flip(dims) if dims else p[j]) / M
                o = moved[1] if moved is not None and moved[0] == t else None
                self.tile(agg[0], t, o).add_(r[0] * self.g)
                self.tile(agg[1], t, o).add_(r[1] * self.g)
                self.tile(wgt, t, o).add_(self.g)
        return agg / wgt, wgt

    def moved_origin(self, t):
        """Tile t's origin moved by one voxel along the first axis where the tile still fits, or None."""
        o = list(self.origins[t])
        for a in range(3):
            for d in (1, -1):
                if 0 <= o[a] + d and o[a] + d + self.ps[a] <= self.shape[a]:
                    o[a] += d
                    return tuple(o)
        return None


def device_call(nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, ranges=((0, -1),)):
    agg = torch.zeros((2,) + tuple(vol.shape), device=vol.device)
    wgt = torch.zeros(tuple(vol.shape), device=vol.device)
    for b, e in ranges:
        nw.accumulate_tiles(vol, agg, wgt, step_size, do_mirroring, mirror_axes, use_gaussian, b, e)
    wgt_acc = wgt.clone()
    seg, p = nw.finalize(agg, wgt)
    return seg, p, wgt_acc


def check_tiling(name, nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, ranges=((0, -1),)):
    seg, p, wgt = device_call(nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, ranges)
    rec = Reconstruction(nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, ranges)
    p_ref, w_ref = rec.aggregate()
    pd = p.double()
    err = (pd - p_ref).abs().max().item()
    sure = (p_ref[1] - p_ref[0]).abs() > SEG_MARGIN
    seg_bad = int((seg.bool() != (p_ref[1] > p_ref[0]))[sure].sum().item())
    wm = nw.weight_map(vol.shape, step_size, use_gaussian).double()
    w_err = max(((wm - w_ref).abs() / w_ref).max().item(), ((wgt.double() - w_ref).abs() / w_ref).max().item())
    def sensitivity(perturbed):
        q, w = perturbed                  # a moved tile can leave a plane without weight: 0 / 0 there
        return (pd - q).abs()[:, w > 0].max().item() / SOFTMAX_TOL

    # the middle tile with one mirror's z-unflip skipped / moved by one voxel
    t = len(rec.origins) // 2
    zs = [j for j, m in enumerate(rec.mirrors) if m & 1]
    o = rec.moved_origin(t)
    sens_z = sensitivity(rec.aggregate(skip_z_unflip=(t, zs[0]))) if zs else None
    sens_o = sensitivity(rec.aggregate(moved=(t, o))) if o is not None else None
    fmt = lambda s: "%9.0f" % s if s is not None else "      n/a"
    print("%-34s tiles %3d x M %d  softmax max|d| %.2e (%.3f of tol)  seg mismatches %d  weight rel %.1e  "
          "sensitivity z-unflip %s origin %s" % (name, len(rec.origins), len(rec.mirrors), err, err / SOFTMAX_TOL, seg_bad,
                                                 w_err, fmt(sens_z), fmt(sens_o)))
    assert err <= SOFTMAX_TOL, (name, err)
    assert seg_bad == 0, (name, seg_bad)
    assert w_err <= WGT_RTOL, (name, w_err)
    for s in (sens_z, sens_o):
        assert s is None or s >= SENS_MIN, (name, sens_z, sens_o)
    return sens_z, sens_o


# ------------------------------------------------------------------------------------------------
# CPU: the reconstruction itself against the oracle's tiled predictor (the oracle network standing in for the device)
# ------------------------------------------------------------------------------------------------
class _OracleForward:
    def __init__(self, net, patch_size):
        self.net, self.patch_size = net, tuple(patch_size)

    def forward_patches(self, x):
        with torch.no_grad():
            return torch.softmax(self.net(x), 1)


@pytest.mark.parametrize("shape,do_mirroring,mirror_axes,step_size", [
    ((40, 50, 45), True, (0, 1, 2), 0.5),
    ((70, 37, 33), True, (0, 2), 0.7),
    ((33, 32, 47), False, (), 0.5),
])
def test_reconstruction_matches_the_oracle_predictor(shape, do_mirroring, mirror_axes, step_size):
    plans = small_plans()
    net = O.build_benchmark_network(0, plans)
    data = O.synthetic_flair(shape, seed=3)
    data[0] = O.zscore_nnunet(data[0], np.where(data[0] != 0, 0, -1), True)
    rec = Reconstruction(_OracleForward(net, (32, 32, 32)), torch.from_numpy(data[0]), step_size, do_mirroring,
                         mirror_axes, True, 8, ((0, 3), (3, -1)))
    p, _ = rec.aggregate()
    _, p_ref = O.predict_3D_tiled(net, data, step_size, do_mirroring, mirror_axes, (32, 32, 32), True)
    assert np.abs(p.numpy() - p_ref).max() < 2e-6


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small_nets():
    """One context of the small plan per max_batch, all with the same weights."""
    import deepwmh_b200
    plans = small_plans()
    net = O.build_benchmark_network(0, plans)
    nets = {}

    def get(max_batch):
        if max_batch not in nets:
            tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=max_batch)
            tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
            nets[max_batch] = tr.network
        return nets[max_batch]
    yield get
    for nw in nets.values():
        nw.close()


def _volume(shape, seed=3):
    data = O.synthetic_flair(shape, seed=seed)
    return torch.from_numpy(O.zscore_nnunet(data[0], np.where(data[0] != 0, 0, -1), True)).cuda()


# (shape, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch)
SMALL_CASES = [
    ((40, 50, 45), 0.5, True, (0, 1, 2), True, 8),
    ((40, 50, 45), 0.7, True, (0, 1, 2), True, 16),
    ((33, 32, 47), 0.5, False, (0, 1, 2), True, 8),
    ((32, 32, 32), 0.5, True, (0, 1, 2), True, 8),            # single tile: no Gaussian
    ((70, 37, 33), 0.5, True, (0, 1, 2), True, 16),           # uneven steps that round
    ((70, 37, 33), 0.7, True, (0, 2), False, 8),
    ((40, 50, 45), 0.5, True, (0, 1), True, 4),               # M = 4 with max_batch 4: one tile per batch
    ((70, 37, 33), 0.7, True, (2,), True, 4),                 # M = 2: two tiles per batch
] + [((33, 32, 47), 0.5, True, axes, True, 8)                 # every mirror subset
     for r in range(4) for axes in itertools.combinations((0, 1, 2), r)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,step_size,do_mirroring,mirror_axes,use_gaussian,max_batch", SMALL_CASES)
def test_tiled_prediction_matches_fp64_aggregation(small_nets, shape, step_size, do_mirroring, mirror_axes, use_gaussian,
                                                   max_batch):
    name = "%s s%.1f %s%s mb%d" % ("x".join(map(str, shape)), step_size, "tta" + "".join(map(str, mirror_axes))
                                   if do_mirroring else "no-tta", "" if use_gaussian else " flat", max_batch)
    check_tiling(name, small_nets(max_batch), _volume(shape), step_size, do_mirroring, mirror_axes, use_gaussian, max_batch)


@pytest.mark.gpu
def test_tile_range_over_two_calls_matches_fp64_aggregation(small_nets):
    vol = _volume((40, 50, 45))
    n = small_nets(8).num_tiles(vol.shape, 0.5)
    sens = check_tiling("40x50x45 tiles [0,5) + [5,%d)" % n, small_nets(8), vol, 0.5, True, (0, 1, 2), True, 8,
                        ((0, 5), (5, -1)))
    assert None not in sens


@pytest.mark.gpu
def test_benchmark_volume_matches_fp64_aggregation():
    """182 x 218 x 182 with the 128^3 plan and 8 mirrors: 12 tiles, 96 forwards, the benchmark's workload."""
    import deepwmh_b200
    plans = deepwmh_b200.benchmark_plans()
    net = O.build_benchmark_network(0, plans)
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=8)
    tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
    try:
        sens = check_tiling("182x218x182 bench tta012 mb8", tr.network, _volume((182, 218, 182), seed=0), 0.5, True,
                            (0, 1, 2), True, 8)
        assert None not in sens
    finally:
        tr.network.close()
