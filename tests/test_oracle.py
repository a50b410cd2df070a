"""CPU: pin the oracle against the known-answer properties of SURVEY.md section 8c (the reference
ships no golden vectors for this path -- `parity unpinned`) and against the committed fixtures."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn as nn
from hypothesis import given, settings, strategies as st

import oracle as O
from conftest import small_plans
from golden import fixtures as F

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_steps_known_answers():
    assert O.compute_steps_for_sliding_window((128,) * 3, (182, 218, 182), 0.5) == [[0, 54], [0, 45, 90], [0, 54]]
    s = O.compute_steps_for_sliding_window((128,) * 3, (512, 512, 320), 0.5)
    assert [len(a) for a in s] == [7, 7, 4]
    assert s[0] == [0, 64, 128, 192, 256, 320, 384] and s[2] == [0, 64, 128, 192]
    assert O.compute_steps_for_sliding_window((128,) * 3, (128,) * 3, 0.5) == [[0], [0], [0]]


@settings(max_examples=200, deadline=None)
@given(patch=st.integers(8, 192), extra=st.integers(0, 400), step=st.sampled_from([0.25, 0.5, 0.75, 1.0, 0.33]))
def test_steps_invariants(patch, extra, step):
    """The four invariants of upstream's tests/test_steps_for_sliding_window_prediction.py (SURVEY.md section 4)."""
    img = patch + extra
    steps = O.compute_steps_for_sliding_window((patch,), (img,), step)[0]
    assert len(steps) == math.ceil((img - patch) / (patch * step)) + 1
    assert steps[0] == 0
    assert steps[-1] + patch == img
    for a, b in zip(steps[:-1], steps[1:]):
        assert 0 < b - a <= math.ceil(patch * step) and b - a <= patch


def test_gaussian_known_answers():
    g = O.get_gaussian((128, 128, 128))
    assert g.dtype == np.float32 and g.max() == 1.0 and np.unravel_index(g.argmax(), g.shape) == (64, 64, 64)
    assert g.min() > 0 and abs(math.log(g.min()) + 24.0) < 0.01          # e^-24 at the far corner
    assert np.array_equal(g[1:], g[1:][::-1]) and np.array_equal(g[:, 1:], g[:, 1:][:, ::-1])
    # separable closed form: exp(-d^2 / (2 sigma^2)) around the centre
    assert abs(g[64, 64, 80] - math.exp(-0.5)) < 1e-6
    g2 = O.get_gaussian((16, 64, 48))
    assert g2.max() == 1.0 and g2.min() > 0


def test_pad_roundtrip():
    x = np.random.default_rng(0).normal(size=(1, 20, 33, 16)).astype(np.float32)
    p, sl = O.pad_nd_image(x, (32, 32, 32))
    assert p.shape == (1, 32, 33, 32)
    assert np.array_equal(p[sl], x)
    assert p[0, :6].sum() == 0 and p[0, 26:].sum() == 0 and sl[1] == slice(6, 26) and sl[3] == slice(8, 24)
    q, sl2 = O.pad_nd_image(x, (8, 8, 8))
    assert q is x and q[sl2].shape == x.shape


def test_network_inventory():
    net = O.build_benchmark_network(0)
    assert O.count_parameters(net) == 31194784
    assert abs(O.forward_flops(O.benchmark_plans()) / 1e9 - 954.46) < 0.01
    keys = set(net.state_dict().keys())
    for k in ["conv_blocks_context.0.blocks.0.conv.weight", "conv_blocks_context.4.blocks.1.instnorm.bias",
              "conv_blocks_context.5.0.blocks.0.conv.weight", "conv_blocks_context.5.1.blocks.0.instnorm.weight",
              "tu.0.weight", "tu.4.weight", "conv_blocks_localization.0.0.blocks.0.conv.weight",
              "conv_blocks_localization.4.1.blocks.0.conv.bias", "seg_outputs.4.weight"]:
        assert k in keys, k
    sd = net.state_dict()
    assert tuple(sd["conv_blocks_localization.0.0.blocks.0.conv.weight"].shape) == (320, 640, 3, 3, 3)
    assert tuple(sd["tu.1.weight"].shape) == (320, 256, 2, 2, 2)
    assert tuple(sd["seg_outputs.4.weight"].shape) == (2, 32, 1, 1, 1)
    assert "seg_outputs.0.bias" not in keys and "tu.0.bias" not in keys


def test_forward_shapes_and_ds(plans_small):
    net = O.build_network(plans_small)
    x = torch.randn(1, 1, 32, 32, 32)
    net.do_ds = True
    outs = net(x)
    assert isinstance(outs, tuple) and outs[0].shape == (1, 2, 32, 32, 32) and outs[1].shape == (1, 2, 16, 16, 16)
    net.do_ds = False
    assert net(x).shape == (1, 2, 32, 32, 32)


def test_conv_bias_cancels_under_instancenorm(plans_small):
    """The CUDA path drops conv biases; exact in real arithmetic, rounding-level here."""
    torch.manual_seed(0)
    net = O.build_benchmark_network(0, plans_small)
    x = torch.randn(1, 1, 32, 32, 32)
    with torch.no_grad():
        y0 = net(x)
        for m in net.modules():
            if isinstance(m, nn.Conv3d) and m.bias is not None:
                m.bias.zero_()
        y1 = net(x)
    assert (y0 - y1).abs().max() < 1e-3


class _ConstNet(O.Generic_UNet):
    def forward(self, x):
        out = torch.zeros(x.shape[0], 2, *x.shape[2:])
        out[:, 1] = 0.7
        return out


class _PointwiseNet(O.Generic_UNet):
    """Mirror-equivariant toy net: logits depend on the voxel value only."""
    def forward(self, x):
        return torch.cat((x, -0.5 * x), 1)


def test_constant_logits_give_constant_output(plans_small):
    net = _ConstNet(1, 32, 2, [[2, 2, 2]] * 3, [[3, 3, 3]] * 4)
    x = np.random.default_rng(1).normal(size=(1, 40, 50, 45)).astype(np.float32)
    seg, p = O.predict_3D(net, x, True, (0, 1, 2), True, 0.5, (32, 32, 32), None, True)
    ref = torch.softmax(torch.tensor([0.0, 0.7]), 0).numpy()
    assert np.allclose(p[0], ref[0], atol=1e-6) and np.allclose(p[1], ref[1], atol=1e-6)
    assert (seg == 1).all() and seg.dtype == np.int64


def test_equivariant_net_tta_equals_no_tta(plans_small):
    net = _PointwiseNet(1, 32, 2, [[2, 2, 2]] * 3, [[3, 3, 3]] * 4)
    x = np.random.default_rng(2).normal(size=(1, 40, 50, 45)).astype(np.float32)
    _, p_tta = O.predict_3D(net, x, True, (0, 1, 2), True, 0.5, (32, 32, 32), None, True)
    _, p_no = O.predict_3D(net, x, False, (0, 1, 2), True, 0.5, (32, 32, 32), None, True)
    assert np.allclose(p_tta, p_no, atol=2e-6)
    expect = torch.softmax(torch.from_numpy(np.concatenate((x, -0.5 * x), 0)), 0).numpy()
    assert np.allclose(p_no, expect, atol=2e-6)


def test_weight_buffer_positive_and_softmax_normalised(plans_small):
    net = O.build_benchmark_network(0, plans_small)
    x = np.random.default_rng(3).normal(size=(1, 45, 40, 50)).astype(np.float32)
    agg, nb = O.predict_3D_tiled(net, x, 0.5, False, (0, 1, 2), (32, 32, 32), True, return_buffers=True)
    assert (nb > 0).all()
    p = agg / nb
    assert np.allclose(p.sum(0), 1.0, atol=1e-5)


def test_small_volume_gets_padded(plans_small):
    net = O.build_benchmark_network(0, plans_small)
    x = np.random.default_rng(4).normal(size=(1, 20, 32, 40)).astype(np.float32)
    seg, p = O.predict_3D(net, x, False, (0, 1, 2), True, 0.5, (32, 32, 32), None, True)
    assert seg.shape == (20, 32, 40) and p.shape == (2, 20, 32, 40)


def test_zscore_variants():
    rng = np.random.default_rng(5)
    v = rng.normal(100, 25, size=(20, 24, 28)).astype(np.float32)
    v[:5] = 0
    seg = np.where(v != 0, 0, -1).astype(np.int8)
    a = O.zscore_nnunet(v, seg, True)
    inside = v != 0
    assert abs(a[inside].mean()) < 1e-5 and abs(a[inside].std() - 1) < 1e-5 and (a[~inside] == 0).all()
    b = O.zscore_nnunet(v, None, False)
    assert abs(b.mean()) < 1e-5 and abs(b.std() - 1) < 1e-4
    c = O.zscore_deepwmh(v, inside.astype(np.float32))       # in-tree sibling: stats over mask, applied everywhere
    assert np.allclose(c[inside], a[inside], atol=1e-5) and not (c[~inside] == 0).any()


def test_synthetic_volume_recipe():
    v = O.synthetic_flair((40, 48, 44), seed=7)
    assert v.shape == (1, 40, 48, 44) and v.dtype == np.float32
    assert v[0, 0, 0, 0] == 0 and v[0, 20, 24, 22] >= 1.0
    assert np.array_equal(v, O.synthetic_flair((40, 48, 44), seed=7))
    assert not np.array_equal(v, O.synthetic_flair((40, 48, 44), seed=8))


def test_dice_definition():
    a = np.zeros((4, 4, 4)); b = np.zeros((4, 4, 4))
    a[:2] = 1; b[1:3] = 1
    assert abs(O.hard_dice_binary(a, b) - 2 * 16 / (32 + 32 + 1e-6)) < 1e-7   # float32 sums, as the reference


@pytest.mark.skipif(not os.path.exists(os.path.join(GOLD, "v1_tta.npz")), reason="fixture not generated")
def test_golden_fixture_consistent_with_oracle_pieces():
    """The committed full-size fixture must agree with cheap pieces of the oracle recomputed now."""
    g = F.load_v1(os.path.join(GOLD, "v1_tta.npz"))
    assert tuple(g["shape"]) == (182, 218, 182)
    raw = O.synthetic_flair((182, 218, 182), seed=0)[0]
    m = raw != 0
    assert np.allclose(g["zscore_mean_std"], [raw[m].mean(), raw[m].std()], rtol=1e-6)
    assert abs(g["seg"].mean() - float(g["fg_frac"][0])) < 1e-9
    seg = np.zeros((182, 218, 182), np.uint8)
    seg[g["seg_sample"]] = g["seg"]
    blk_sample = g["seg_sample"][F.V1_BLOCK]
    assert np.array_equal(seg[F.V1_BLOCK][blk_sample], (g["p1_block"] > g["p0_block"]).astype(np.uint8)[blk_sample])
    assert np.allclose(g["p1_block"] + g["p0_block"], 1.0, atol=1e-5)
