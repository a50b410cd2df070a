"""GPU (plain torch, TF32 off): full-volume parity-gate numbers of rounding-point VARIANTS of the fp16 scheme,
against the fp32 oracle, to decide where extra precision pays.  Test infrastructure (imports oracle/).

usage: python tools/precision_full.py variant [variant ...]
  variants: base | lastfp32 (last conv output kept fp32) | last2fp32 | storefp32 (all raw outputs fp32)
            | skipfp32 (skip tensors kept fp32 for the decoder concat)
"""
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle as O  # noqa: E402
from golden import fixtures as GF  # noqa: E402

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
H = torch.float16


def rnd(x, on=True):
    return x.to(H).to(torch.float32) if on else x


def rnd_dither(x):
    """unbiased (stochastic) rounding to fp16: add uniform noise of +-0.5 ulp, then round to nearest"""
    ulp = torch.pow(2.0, torch.floor(torch.log2(x.abs().clamp_min(6.2e-5))) - 10)
    return (x + (torch.rand_like(x) - 0.5) * ulp).to(H).to(torch.float32)


_WCACHE = {}


def rnd_w_diffused(w):
    """sum-preserving rounding of conv weights: the rounding residual is carried from tap to tap, so the DC gain
    sum_taps w[co,ci,:] of every (co,ci) filter is exact to one fp16 ulp (constant regions see only the DC gain)"""
    key = id(w)
    if key not in _WCACHE:
        flat = w.detach().reshape(w.shape[0], w.shape[1], -1).double()
        out = torch.empty_like(flat)
        r = torch.zeros_like(flat[..., 0])
        for t in range(flat.shape[-1]):
            q = (flat[..., t] + r).to(H).double()
            r = flat[..., t] + r - q
            out[..., t] = q
        _WCACHE[key] = out.float().reshape(w.shape)
    return _WCACHE[key]


RES32 = [0]   # raw outputs with spatial edge <= RES32[0] are kept fp32


def block(blk, x, first, store16, op16=True, wdiff=False, dither_x=False, dither_y=False):
    w = blk.conv.weight if first else (rnd_w_diffused(blk.conv.weight) if wdiff else rnd(blk.conv.weight, op16))
    xin = x if first else (rnd_dither(x) if dither_x else rnd(x, op16))
    y = F.conv3d(xin, w, None, blk.conv.stride, blk.conv.padding)
    mean = y.mean(dim=(2, 3, 4), keepdim=True)
    var = y.var(dim=(2, 3, 4), keepdim=True, unbiased=False)
    a = blk.instnorm.weight.view(1, -1, 1, 1, 1) / torch.sqrt(var + 1e-5)
    b = blk.instnorm.bias.view(1, -1, 1, 1, 1) - mean * a
    if y.shape[-1] <= RES32[0]:
        store16 = False
    ys = rnd_dither(y) if (dither_y and store16) else rnd(y, store16)
    return F.leaky_relu(a * ys + b, 0.01)


class Emu(torch.nn.Module):
    def __init__(self, net, variant):
        super().__init__()
        self.net, self.variant = net, variant
        self.num_classes = 2
        self._gaussian_3d = None
        self._patch_size_for_gaussian_3d = None
        self.inference_apply_nonlin = lambda x: F.softmax(x, 1)

    def forward(self, x):
        net, v = self.net, self.variant
        blocks = []
        for d in range(len(net.conv_blocks_context) - 1):
            blocks += [("enc", d, b) for b in net.conv_blocks_context[d].blocks]
        nconv = 2 * len(net.conv_blocks_context) + 2 * len(net.tu)
        ci = 0
        skips = []

        def store16(idx):
            if v == "storefp32":
                return False
            if v == "lastfp32" and idx == nconv - 1:
                return False
            if v == "last2fp32" and idx >= nconv - 2:
                return False
            return True
        kw = dict(wdiff='wdiff' in v, dither_x='dx' in v, dither_y='dy' in v)
        first = True
        for d in range(len(net.conv_blocks_context) - 1):
            for blk in net.conv_blocks_context[d].blocks:
                x = block(blk, x, first, store16(ci), **kw); first = False; ci += 1
            skips.append(x)
        for st in net.conv_blocks_context[-1]:
            for blk in st.blocks:
                x = block(blk, x, False, store16(ci), **kw); ci += 1
        for u in range(len(net.tu)):
            up = rnd(F.conv_transpose3d(rnd(x), rnd(net.tu[u].weight), None, net.tu[u].stride))
            x = torch.cat((up, skips[-(u + 1)]), 1)
            for st in net.conv_blocks_localization[u]:
                for blk in st.blocks:
                    x = block(blk, x, False, store16(ci), **kw); ci += 1
        return net.seg_outputs[-1](x)


def predict(net_like, data, patch=(128, 128, 128)):
    steps = O.compute_steps_for_sliding_window(patch, data.shape[1:], 0.5)
    g = torch.from_numpy(O.get_gaussian(patch)).cuda()
    agg = torch.zeros((2,) + data.shape[1:], device="cuda"); nb = torch.zeros(data.shape[1:], device="cuda")
    vol = torch.from_numpy(data).cuda()
    with torch.no_grad():
        for lx in steps[0]:
            for ly in steps[1]:
                for lz in steps[2]:
                    t = vol[None, :, lx:lx + 128, ly:ly + 128, lz:lz + 128]
                    acc = torch.zeros(1, 2, 128, 128, 128, device="cuda")
                    for m in range(8):
                        dims = O.MIRROR_DIMS[m]
                        xin = torch.flip(t, dims) if dims else t
                        p = F.softmax(net_like(xin.contiguous()), 1)
                        acc += 1 / 8 * (torch.flip(p, dims) if dims else p)
                    agg[:, lx:lx + 128, ly:ly + 128, lz:lz + 128] += acc[0] * g
                    nb[lx:lx + 128, ly:ly + 128, lz:lz + 128] += g
    p = (agg / nb).cpu().numpy()
    return p.argmax(0), p


def main():
    variants = sys.argv[1:] or ["base"]
    net = O.build_benchmark_network(0).cuda()
    raw = O.synthetic_flair(seed=0)
    data = raw.copy()
    data[0] = O.zscore_nnunet(raw[0], np.where(raw[0] != 0, 0, -1), True)
    t0 = time.time()
    seg_r, p_r = predict(net, data)
    print("fp32 oracle on GPU: %.1fs, fg=%.4f" % (time.time() - t0, seg_r.mean()))
    gpath = os.path.join(ROOT, "tests", "golden", "v1_tta.npz")
    if os.path.exists(gpath):
        g = GF.load_v1(gpath)               # the argmax of a seeded half of the voxels
        print("GPU fp32 oracle vs committed CPU golden: agree %.6f" % np.mean(g["seg"] == seg_r[g["seg_sample"]]))
    head = raw[0] != 0
    print("near-boundary mass: frac |p-0.5|<1e-3: all %.5f  head %.5f  background %.5f" % (
        np.mean(np.abs(p_r[1] - 0.5) < 1e-3), np.mean(np.abs(p_r[1][head] - 0.5) < 1e-3), np.mean(np.abs(p_r[1][~head] - 0.5) < 1e-3)))
    for v in variants:
        RES32[0] = int(v[2:]) if v.startswith("le") else 0
        seg, p = predict(Emu(net, v), data)
        rep = O.parity_report(seg_r, p_r, seg, p)
        flips = seg != seg_r
        print("%-10s agree %.6f dice %.6f softmax|d| max %.3e mean %.3e | flips in head %.6f background %.6f" % (
            v, rep["argmax_agree"], rep["dice"], rep["softmax_max_abs"], np.abs(p - p_r).mean(), flips[head].mean(), flips[~head].mean()))


if __name__ == "__main__":
    main()
