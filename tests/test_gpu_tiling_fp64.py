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
weights and the mirror average.  Perturbed references of the middle tile -- one mirror's z-unflip skipped, the origin
moved by a voxel, its forwards run with modalities 0 and 1 exchanged (M > 1), its mirrors read with the two-class stride
(C > 2) -- must each differ from the device result by 100 times the tolerance, which shows that each would be caught.

Volumes are [M, X, Y, Z] for M modalities ([X, Y, Z] for one) and the result has C classes: the cases with M > 1 reach
the first conv's tile fetch with a modality stride (the tcgen05 kernel on the cube plan, conv_first_kernel on the
anisotropic one), and each class count reaches the overlap-add and finalize instantiated for it.  A single tile with one
mirror axis is also checked bit for bit against its two forwards.
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


def _lead(vol):
    """A [X, Y, Z] volume (one modality) as [1, X, Y, Z]; [M, X, Y, Z] as it is."""
    return vol if vol.dim() == 4 else vol[None]


class Reconstruction:
    """The device's tiled call restated on the host: forwards through `forward_patches`, everything else in float64.
    vol: [M, X, Y, Z] (or [X, Y, Z] for one modality); C = nw.num_classes."""

    def __init__(self, nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, ranges=((0, -1),)):
        ps = tuple(nw.patch_size)
        vol = _lead(vol)
        steps = O.compute_steps_for_sliding_window(ps, vol.shape[1:], step_size)
        self.nw, self.vol = nw, vol
        self.ps, self.shape = ps, tuple(vol.shape[1:])
        self.origins = [(x, y, z) for x in steps[0] for y in steps[1] for z in steps[2]]
        self.mirrors = mirror_list(do_mirroring, mirror_axes)
        nm = len(self.mirrors)
        per_batch = max(1, max_batch // nm)
        if use_gaussian and len(self.origins) > 1:
            self.g = torch.from_numpy(O.get_gaussian(ps)).to(vol.device, torch.float64)
        else:
            self.g = torch.ones(ps, dtype=torch.float64, device=vol.device)
        self.probs = {}                   # tile index -> the mirrored forwards as [mirrors, C, *patch] fp64, still flipped
        for b, e in ranges:
            e = len(self.origins) if e < 0 else e
            for t0 in range(b, e, per_batch):
                tiles = range(t0, min(t0 + per_batch, e))
                p = self.forwards(tiles)
                for k, t in enumerate(tiles):
                    self.probs.setdefault(t, []).append(p[k * nm:(k + 1) * nm])

    def forwards(self, tiles, swap_modalities=False):
        """One forward_patches call over the mirrored tiles (modalities 0 and 1 exchanged when swap_modalities)."""
        vol = self.vol[[1, 0] + list(range(2, self.vol.shape[0]))] if swap_modalities else self.vol
        patches = torch.stack([self.tile(vol, t).flip(flip_dims(m, 1)) for t in tiles for m in self.mirrors])
        return self.nw.forward_patches(patches.contiguous()).double()

    def tile(self, vol, t, origin=None):
        """Tile t of the last three axes of vol."""
        o = self.origins[t] if origin is None else origin
        return vol[..., o[0]:o[0] + self.ps[0], o[1]:o[1] + self.ps[1], o[2]:o[2] + self.ps[2]]

    def aggregate(self, skip_z_unflip=None, moved=None, replaced=None, two_class_stride=None):
        """(softmax, weight sum) in float64.  Perturbations of one tile t: skip_z_unflip = (t, mirror index) leaves that
        forward's z axis flipped; moved = (t, origin) adds the tile at another origin; replaced = (t, forwards) uses other
        forwards for it; two_class_stride = t reads class c of mirror j from [(j * 2 + c) * P] of the tile's [mirrors][C][P]
        block, the indexing of a two-class overlap-add."""
        dev = self.g.device
        C = self.nw.num_classes
        agg = torch.zeros((C,) + self.shape, dtype=torch.float64, device=dev)
        wgt = torch.zeros(self.shape, dtype=torch.float64, device=dev)
        nm = len(self.mirrors)
        for t, parts in self.probs.items():
            for p in parts:                       # one entry per call that covered the tile
                if replaced is not None and replaced[0] == t:
                    p = replaced[1]
                if two_class_stride == t:
                    flat = p.reshape(nm * C, -1)
                    p = torch.stack([torch.stack([flat[j * 2 + c] for c in range(C)]) for j in range(nm)]).view(p.shape)
                r = torch.zeros((C,) + self.ps, dtype=torch.float64, device=dev)
                for j, m in enumerate(self.mirrors):
                    dims = flip_dims(m, 1)
                    if skip_z_unflip == (t, j):
                        dims = [d for d in dims if d != 3]
                    r += (p[j].flip(dims) if dims else p[j]) / nm
                o = moved[1] if moved is not None and moved[0] == t else None
                self.tile(agg, t, o).add_(r * self.g)
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
    shape = tuple(vol.shape[-3:])
    agg = torch.zeros((nw.num_classes,) + shape, device=vol.device)
    wgt = torch.zeros(shape, device=vol.device)
    for b, e in ranges:
        nw.accumulate_tiles(vol, agg, wgt, step_size, do_mirroring, mirror_axes, use_gaussian, b, e)
    wgt_acc = wgt.clone()
    seg, p = nw.finalize(agg, wgt)
    return seg, p, wgt_acc


def label_mismatches(seg, p_ref):
    """Voxels whose device label is not the reference's argmax, counted where the reference's top-two margin exceeds
    SEG_MARGIN (closer calls may go either way under fp32 rounding)."""
    top = p_ref.topk(2, dim=0).values
    sure = (top[0] - top[1]) > SEG_MARGIN
    return int((seg.long() != p_ref.argmax(0))[sure].sum().item())


def check_tiling(name, nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, ranges=((0, -1),)):
    seg, p, wgt = device_call(nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, ranges)
    rec = Reconstruction(nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, ranges)
    p_ref, w_ref = rec.aggregate()
    pd = p.double()
    err = (pd - p_ref).abs().max().item()
    seg_bad = label_mismatches(seg, p_ref)
    wm = nw.weight_map(rec.shape, step_size, use_gaussian).double()
    w_err = max(((wm - w_ref).abs() / w_ref).max().item(), ((wgt.double() - w_ref).abs() / w_ref).max().item())
    def sensitivity(perturbed):
        q, w = perturbed                  # a moved tile can leave a plane without weight: 0 / 0 there
        return (pd - q).abs()[:, w > 0].max().item() / SOFTMAX_TOL

    # the middle tile with one mirror's z-unflip skipped / moved by one voxel / its forwards with modalities 0 and 1
    # exchanged (M > 1) / its mirrors read with the two-class stride (C > 2)
    t = len(rec.origins) // 2
    zs = [j for j, m in enumerate(rec.mirrors) if m & 1]
    o = rec.moved_origin(t)
    sens = {"z-unflip": sensitivity(rec.aggregate(skip_z_unflip=(t, zs[0]))) if zs else None,
            "origin": sensitivity(rec.aggregate(moved=(t, o))) if o is not None else None,
            "modality": sensitivity(rec.aggregate(replaced=(t, rec.forwards([t], swap_modalities=True))))
            if rec.vol.shape[0] > 1 else None,
            # (with one mirror the two strides read the same elements)
            "class-stride": sensitivity(rec.aggregate(two_class_stride=t)) if nw.num_classes > 2 and len(rec.mirrors) > 1
            else None}
    fmt = lambda s: "%9.0f" % s if s is not None else "      n/a"
    print("%-40s tiles %3d x mirrors %d  softmax max|d| %.2e (%.3f of tol)  seg mismatches %d  weight rel %.1e  "
          "sensitivity %s" % (name, len(rec.origins), len(rec.mirrors), err, err / SOFTMAX_TOL, seg_bad, w_err,
                              " ".join("%s %s" % (k, fmt(v)) for k, v in sens.items())))
    assert err <= SOFTMAX_TOL, (name, err)
    assert seg_bad == 0, (name, seg_bad)
    assert w_err <= WGT_RTOL, (name, w_err)
    for s in sens.values():
        assert s is None or s >= SENS_MIN, (name, sens)
    return sens


# ------------------------------------------------------------------------------------------------
# CPU: the reconstruction itself against the oracle's tiled predictor (the oracle network standing in for the device)
# ------------------------------------------------------------------------------------------------
class _OracleForward:
    def __init__(self, net, patch_size):
        self.net, self.patch_size = net, tuple(patch_size)
        self.num_classes = net.num_classes

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


def test_reconstruction_with_two_modalities_and_three_classes_matches_the_oracle_predictor():
    from test_gpu_multimodal import _plans
    plans = _plans("cube", 2, 3)
    net = O.build_benchmark_network(0, plans)
    data = _volume_np((40, 50, 45), 2)
    rec = Reconstruction(_OracleForward(net, (32, 32, 32)), torch.from_numpy(data), 0.5, True, (0, 1, 2), True, 8,
                         ((0, 3), (3, -1)))
    p, _ = rec.aggregate()
    assert p.shape == (3, 40, 50, 45)
    _, p_ref = O.predict_3D_tiled(net, data, 0.5, True, (0, 1, 2), (32, 32, 32), True)
    assert np.abs(p.numpy() - p_ref).max() < 2e-6


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small_nets():
    """One context per (plan, modalities, classes, max_batch); the weights depend only on the first three."""
    import deepwmh_b200
    from test_gpu_multimodal import _plans
    nets, weights = {}, {}

    def get(max_batch, kind="cube", M=1, C=2):
        key = (kind, M, C)
        if key not in weights:
            plans = small_plans() if key == ("cube", 1, 2) else _plans(kind, M, C)
            weights[key] = (plans, O.build_benchmark_network(0, plans).state_dict())
        if key + (max_batch,) not in nets:
            plans, sd = weights[key]
            tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=max_batch)
            tr.load_checkpoint_ram({"state_dict": sd}, False)
            nets[key + (max_batch,)] = tr.network
        return nets[key + (max_batch,)]
    yield get
    for nw in nets.values():
        nw.close()


def _volume_np(shape, M=1, seed=3):
    """M z-scored synthetic volumes [M, X, Y, Z] (modality m from seed + m); zero background shared by none."""
    out = np.empty((M,) + tuple(shape), np.float32)
    for m in range(M):
        data = O.synthetic_flair(shape, seed=seed + m)
        out[m] = O.zscore_nnunet(data[0], np.where(data[0] != 0, 0, -1), True)
    return out


def _volume(shape, seed=3, M=None):
    """[X, Y, Z] on the device (M None: the single-modality tests' volume) or [M, X, Y, Z]."""
    v = torch.from_numpy(_volume_np(shape, M or 1, seed)).cuda()
    return v if M is not None else v[0]


# (shape, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, plan, modalities, classes, tile ranges)
ALL = (0, 1, 2)
SMALL_CASES = [
    ((40, 50, 45), 0.5, True, ALL, True, 8),
    ((40, 50, 45), 0.7, True, ALL, True, 16),
    ((33, 32, 47), 0.5, False, ALL, True, 8),
    ((32, 32, 32), 0.5, True, ALL, True, 8),                  # single tile: no Gaussian
    ((70, 37, 33), 0.5, True, ALL, True, 16),                 # uneven steps that round
    ((70, 37, 33), 0.7, True, (0, 2), False, 8),
    ((40, 50, 45), 0.5, True, (0, 1), True, 4),               # M = 4 with max_batch 4: one tile per batch
    ((70, 37, 33), 0.7, True, (2,), True, 4),                 # M = 2: two tiles per batch
] + [((33, 32, 47), 0.5, True, axes, True, 8)                 # every mirror subset
     for r in range(4) for axes in itertools.combinations(ALL, r)]
SMALL_IDS = ["shape%d-%s-%s-mirror_axes%d-%s-%d" % (i, c[1], c[2], i, c[4], c[5]) for i, c in enumerate(SMALL_CASES)]
SMALL_CASES = [c + ("cube", 1, 2, ((0, -1),)) for c in SMALL_CASES]
# several modalities (the first conv's tile fetch with a modality stride) and classes (aggregate_tile_kernel<C>,
# finalize_kernel<C, VEC>); (3, 2) feeds three modalities to the two-class overlap-add
MC_CASES = [((40, 50, 45), 0.5, True, ALL, True, 8, "cube", M, C, ((0, -1),)) for M, C in ((2, 3), (4, 4), (3, 2), (1, 8))] + [
    ((24, 70, 60), 0.5, True, ALL, True, 8, "aniso", 2, 3, ((0, -1),)),      # the CUDA-core first conv in tile mode
    ((40, 50, 45), 0.5, True, (0, 1), True, 4, "cube", 2, 3, ((0, -1),)),    # one tile per batch
    ((40, 50, 45), 0.7, True, ALL, True, 16, "cube", 2, 3, ((0, -1),)),      # two tiles per batch
    ((40, 50, 45), 0.5, True, ALL, True, 8, "cube", 2, 3, ((0, 5), (5, -1))),   # a tile range over two calls
    ((35, 33, 37), 0.5, True, ALL, True, 8, "cube", 2, 3, ((0, -1),)),      # X Y Z % 4 != 0: unaligned modality stride
] + [((33, 32, 47), 0.5, True, axes, True, 8, "cube", 2, 3, ((0, -1),))     # every mirror subset
     for r in range(4) for axes in itertools.combinations(ALL, r)]


def _case_name(shape, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, kind, M, C, ranges):
    return "%s%s s%.1f %s%s mb%d%s" % (
        "" if (kind, M, C) == ("cube", 1, 2) else "%s M%d C%d " % (kind, M, C), "x".join(map(str, shape)), step_size,
        "tta" + "".join(map(str, mirror_axes)) if do_mirroring else "no-tta", "" if use_gaussian else " flat", max_batch,
        "" if ranges == ((0, -1),) else " tiles " + "+".join("%d:%s" % (b, e if e >= 0 else "end") for b, e in ranges))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,step_size,do_mirroring,mirror_axes,use_gaussian,max_batch,kind,M,C,ranges",
                         SMALL_CASES + MC_CASES, ids=SMALL_IDS + [_case_name(*c).replace(" ", "-") for c in MC_CASES])
def test_tiled_prediction_matches_fp64_aggregation(small_nets, shape, step_size, do_mirroring, mirror_axes, use_gaussian,
                                                   max_batch, kind, M, C, ranges):
    name = _case_name(shape, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, kind, M, C, ranges)
    nw = small_nets(max_batch, kind, M, C)
    vol = _volume(shape, M=M) if M > 1 else _volume(shape)
    sens = check_tiling(name, nw, vol, step_size, do_mirroring, mirror_axes, use_gaussian, max_batch, ranges)
    if M > 1:
        assert sens["modality"] is not None
    if C > 2 and len(mirror_list(do_mirroring, mirror_axes)) > 1:
        assert sens["class-stride"] is not None


@pytest.mark.gpu
def test_tile_range_over_two_calls_matches_fp64_aggregation(small_nets):
    vol = _volume((40, 50, 45))
    n = small_nets(8).num_tiles(vol.shape, 0.5)
    sens = check_tiling("40x50x45 tiles [0,5) + [5,%d)" % n, small_nets(8), vol, 0.5, True, (0, 1, 2), True, 8,
                        ((0, 5), (5, -1)))
    assert sens["z-unflip"] is not None and sens["origin"] is not None


@pytest.mark.gpu
@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("kind,M,C", [("cube", 2, 3), ("cube", 4, 4), ("aniso", 2, 3), ("aniso", 4, 4)])
def test_single_tile_is_the_exact_mirror_mean_of_its_forwards(small_nets, kind, M, C, axis):
    """A volume of the patch's size mirrored along one axis: one tile, two forwards, no Gaussian.  The overlap-add then
    is 0.5 p0 + 0.5 unflip(p1) with both products exact and one rounding, in any fp32 order -- so the device's tile
    (fetcher: modality stride, flip of that axis; aggregate: unflip) must equal, bit for bit, that sum formed from one
    forward_patches call on the same two-sample batch.  Voxels where p0 or p1 is not a normal fp32 number are left out:
    there flush-to-zero or a contracted multiply-add may change the last bit."""
    nw = small_nets(8, kind, M, C)
    vol = _volume(nw.patch_size, M=M)
    d = 1 + axis
    p = nw.forward_patches(torch.stack([vol, vol.flip(d)]).contiguous())
    p0, p1 = p[0], p[1].flip(d)
    want = 0.5 * p0 + 0.5 * p1
    agg = torch.zeros((C,) + tuple(nw.patch_size), device="cuda")
    wgt = torch.zeros(tuple(nw.patch_size), device="cuda")
    nw.accumulate_tiles(vol, agg, wgt, 0.5, True, (axis,), True)
    tiny = torch.finfo(torch.float32).tiny
    normal = (p0.abs() >= tiny) & (p1.abs() >= tiny)
    bad = int((agg != want)[normal].sum().item())
    print("%s M=%d C=%d mirror axis %d: %d of %d values differ, %d left out (not normal)"
          % (kind, M, C, axis, bad, normal.numel(), int((~normal).sum().item())))
    assert torch.equal(wgt, torch.ones_like(wgt))
    assert bad == 0
    # the mirror does matter: without the unflip the sum is another one
    assert not torch.equal(agg, 0.5 * p0 + 0.5 * p[1])


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
        assert sens["z-unflip"] is not None and sens["origin"] is not None
    finally:
        tr.network.close()
