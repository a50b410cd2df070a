"""Every layer of the device network against a float64 reference that is fed exactly what the device layer was fed.

The reference is the oracle network in float64 with the device's weight rounding (`dwmh_commit_weights`: every conv but
the first and every transposed conv rounded to the activation type; the first conv kept in fp32, which its hi + lo split
reproduces to about 2^-22; conv biases dropped, they cancel under InstanceNorm).  A forward hook on every
ConvDropoutNormNonlin and ConvTranspose3d keeps the module's float64 output as that layer's reference and hands the
device's own output of the same layer to everything downstream, the skip concatenations included.  So errors do not pile
up along the network: what is left at each layer is that kernel's own rounding, and it is bounded per element by a
rounding model instead of a fraction of the layer maximum.

Per element, with y the float64 raw conv output, sigma = sqrt(var(y) + 1e-5) per sample and channel, A = conv(|x|, |w|)
and u the unit roundoff of the activation type (2^-11 fp16, 2^-8 bf16):

    conv + InstanceNorm + LeakyReLU   |dev - ref| <= 2u|ref| + s (|gamma| / sigma)(eps_raw |y| + 2^-14 A) + 2^-24
    transposed conv                   |dev - ref| <= 2u|ref| + 2^-14 A
    head (1x1x1 + softmax)            |p_dev - p_ref| <= 1e-6 + 2^-14 sum_k A_k    (A_k: the logit of class k on |x|, |w|)

eps_raw = u where the raw conv output is stored in the activation type (the first conv, the last conv and every layer
with an edge above 64 voxels) and 2^-23 where it is kept in fp32.  2u|ref| covers the output rounding, 2^-14 A the fp32
accumulation over up to 27 * 640 products (random-sign errors, a bound that is loose by the square root of that count).
s is the LeakyReLU's slope at the reference: 0.01 where the reference pre-activation lies below minus the error term,
1 elsewhere.  The activation scales the error of its input by its slope.  Without s the elements on the negative side
(about half of them) get a tolerance 100x too wide, the median of the sensitivity check below lands between the two
halves, and it drops to 4.2 on the 128-channel decoder conv of the 32^3 plan already (CPU emulation); with s it is 49.

A tolerance is only worth something if it can see a wrong kernel.  Each layer therefore also recomputes its reference
with one piece of the operation removed -- the centre tap of every input channel for a conv, one of the output parity
classes for a transposed conv -- and requires the median of |perturbed - ref| / tol to be at least 4 (on the affected
elements).  The head's reference is recomputed with the last class's weights of channels 0-3 and 4-7 exchanged -- the
error of a coefficient chunk index that is off by one -- and the median over that class must reach the same 4.  Only the
host reference is perturbed.

The GPU cases reach the kernel paths DESIGN section 4 describes; the CPU test runs the same harness against an emulation
of the device's fp16 scheme, which pins the tolerance model and the hook plumbing without a GPU.
"""
import copy

import pytest
import torch
import torch.nn.functional as F

import oracle as O
from conftest import small_plans

U = {"fp16": 2.0 ** -11, "bf16": 2.0 ** -8}
SENS_MIN = 4.0
RAW32_MAX_EDGE = 64    # mirrors RAW32_MAX_EDGE in csrc/api.cu: the largest edge whose raw conv output is stored in fp32


def round_act(t, act):
    """Round to the activation type (fp16 or bf16, round to nearest even) and back to t's dtype."""
    return t.to(torch.float16 if act == "fp16" else torch.bfloat16).to(t.dtype)


def _first_conv(net):
    return net.conv_blocks_context[0].blocks[0]


def _last_conv(net):
    return net.conv_blocks_localization[-1][-1].blocks[-1]


def _sub(t, cap=1 << 22):
    """A fixed, evenly strided subset of at most ~cap elements (medians of 10^8-element tensors)."""
    t = t.reshape(-1)
    return t[::max(1, t.numel() // cap)]


def rounded_copy(net, act, dtype, device):
    """The oracle network with the device's weight rounding, in `dtype` on `device`."""
    ref = copy.deepcopy(net).to(device=device, dtype=dtype).eval()
    first = _first_conv(ref)
    with torch.no_grad():
        for m in ref.modules():
            if isinstance(m, O.ConvDropoutNormNonlin):
                m.conv.bias.zero_()
                if m is not first:
                    m.conv.weight.copy_(round_act(m.conv.weight, act))
            elif isinstance(m, torch.nn.ConvTranspose3d):
                m.weight.copy_(round_act(m.weight, act))
    return ref


def _instnorm_lrelu(y, m):
    return F.leaky_relu(F.instance_norm(y, weight=m.instnorm.weight, bias=m.instnorm.bias, eps=1e-5), 1e-2)


def conv_report(m, x, y, ref, dev, u, eps_raw):
    """max |dev - ref| / tol and the sensitivity ratio of one conv + InstanceNorm + LeakyReLU layer."""
    conv = m.conv
    w = conv.weight
    a = F.conv3d(x.abs(), w.abs(), None, conv.stride, conv.padding)
    var = y.var(dim=(2, 3, 4), unbiased=False, keepdim=True)
    g = m.instnorm.weight.abs().view(1, -1, 1, 1, 1) / torch.sqrt(var + 1e-5)
    e = g * (eps_raw * y.abs() + 2.0 ** -14 * a)
    # the LeakyReLU passes an error of its input on with its slope: 0.01 where the pre-activation stays negative
    slope = torch.where(torch.where(ref > 0, ref, ref * 100.0) > -e, 1.0, 1e-2)
    tol = 2 * u * ref.abs() + slope * e + 2.0 ** -24
    err = ((dev - ref).abs() / tol).max().item()
    # the same layer without the centre tap of every input channel (a 1x1x1 conv with the layer's stride)
    c = tuple(k // 2 for k in w.shape[2:])
    yc = F.conv3d(x, w[:, :, c[0], c[1], c[2]][..., None, None, None], None, conv.stride)
    sens = torch.median(_sub((_instnorm_lrelu(y - yc, m) - ref).abs() / tol)).item()
    return err, sens


def tconv_report(m, x, ref, dev, u):
    a = F.conv_transpose3d(x.abs(), m.weight.abs(), None, m.stride)
    tol = 2 * u * ref.abs() + 2.0 ** -14 * a
    err = ((dev - ref).abs() / tol).max().item()
    # output parity class (0, 0, 0) dropped: there the perturbed reference is 0
    par = (slice(None), slice(None)) + tuple(slice(0, None, s) for s in m.stride)
    sens = torch.median(_sub(ref[par].abs() / tol[par])).item()
    return err, sens


def swap_last_class_chunks(w):
    """The head weights [C, c, 1, 1, 1] with the last class's channels 0-3 and 4-7 exchanged: what the two-voxel head
    computes if its float4 coefficient index (k * 8 + cc * 2 + h) is off by one chunk for that class."""
    w = w.clone()
    w[-1, 0:8] = torch.cat([w[-1, 4:8], w[-1, 0:4]])
    return w


def head_report(net, last, probs):
    """max |p_dev - p_ref| / tol of the head, and the median of |p_swapped - p_ref| / tol over the last class, with
    p_swapped the reference computed from swap_last_class_chunks's weights."""
    w = net.seg_outputs[-1].weight
    p_ref = torch.softmax(F.conv3d(last, w), 1)
    a = F.conv3d(last.abs(), w.abs()).sum(1, keepdim=True)
    tol = 1e-6 + 2.0 ** -14 * a
    p_swap = torch.softmax(F.conv3d(last, swap_last_class_chunks(w)), 1)
    sens = torch.median(_sub((p_swap - p_ref)[:, -1:].abs() / tol)).item()
    return ((probs - p_ref).abs() / tol).max().item(), sens


def layer_fp64_reports(net, dev, x, act="fp16", ref_device=None, samples=None):
    """Run `dev` (a SegmentationNetwork, or the CPU emulation below) on x [n, 1, *patch] and compare each of its layers with
    the float64 reference fed the device's previous outputs.  Returns one dict per device layer, in device order (the
    execution order of the network), and the head's (ratio, sensitivity).  samples: check only these samples of the batch
    (the device still runs all n; InstanceNorm is per sample, so each sample's layers are independent of the others)."""
    ref_device = ref_device if ref_device is not None else x.device
    n, u = x.shape[0], U[act]
    probs = dev.forward_patches(x)
    if samples is None:
        fetch = lambda i: dev.layer_output(i, n)
    else:
        samples = list(samples)
        probs, x = probs[samples], x[samples]
        fetch = lambda i: dev.layer_output(i, samples=samples)
    probs = probs.to(ref_device, torch.float64)
    ref_net = rounded_copy(net, act, torch.float64, ref_device)
    first, last = _first_conv(ref_net), _last_conv(ref_net)
    reports, raw, hooks = [], {}, []

    def on_conv(mod, inp, out):
        raw[mod] = out

    def on_layer(mod, inp, out):
        i = len(reports)
        x_in = inp[0]
        got = fetch(i).to(ref_device, torch.float64)
        assert got.shape == out.shape, (i, tuple(got.shape), tuple(out.shape))
        rep = {"layer": i, "shape": tuple(out.shape[1:]), "norm_on_load": dev.layer_norm_on_load(i) == 1}
        if isinstance(mod, O.ConvDropoutNormNonlin):
            edge = max(out.shape[2:])
            eps_raw = u if (mod is first or mod is last or edge > RAW32_MAX_EDGE) else 2.0 ** -23
            rep["kind"] = "conv s%s k%s" % ("".join(map(str, mod.conv.stride)), "".join(map(str, mod.conv.kernel_size)))
            rep["err"], rep["sens"] = conv_report(mod, x_in, raw.pop(mod.conv), out, got, u, eps_raw)
        else:
            rep["kind"] = "tconv s%s" % "".join(map(str, mod.stride))
            rep["err"], rep["sens"] = tconv_report(mod, x_in, out, got, u)
        reports.append(rep)
        # a producer normalised on load is rounded to the activation type by its consumer's loader, not before
        return round_act(got, act) if rep["norm_on_load"] else got

    for m in ref_net.modules():
        if isinstance(m, O.ConvDropoutNormNonlin):
            hooks.append(m.conv.register_forward_hook(on_conv))
            hooks.append(m.register_forward_hook(on_layer))
        elif isinstance(m, torch.nn.ConvTranspose3d):
            hooks.append(m.register_forward_hook(on_layer))
    try:
        with torch.no_grad():
            ref_net(x.to(ref_device, torch.float64))
            assert len(reports) == dev.num_layers(), (len(reports), dev.num_layers())
            head = head_report(ref_net, fetch(len(reports) - 1).to(ref_device, torch.float64), probs)
    finally:
        for h in hooks:
            h.remove()
    return reports, head


def print_reports(name, reports, head):
    for r in reports:
        print("%-22s layer %2d %-12s %-18s%s max err/tol %.3f  sensitivity %8.1f" % (
            name, r["layer"], r["kind"], "x".join(map(str, r["shape"])), " nol" if r["norm_on_load"] else "    ",
            r["err"], r["sens"]))
    print("%-22s head                                  max err/tol %.3f  sensitivity %8.1f" % ((name,) + head))


def check_reports(name, reports, head):
    """head: (max err/tol, sensitivity) of head_report."""
    print_reports(name, reports, head)
    bad = [(r["layer"], r["kind"], round(r["err"], 3)) for r in reports if not r["err"] <= 1.0]
    blind = [(r["layer"], r["kind"], round(r["sens"], 2)) for r in reports if not r["sens"] >= SENS_MIN]
    assert not bad, (name, "above tolerance", bad)
    assert not blind, (name, "tolerance cannot see a one-tap error", blind)
    assert head[0] <= 1.0, (name, "head", head)
    assert head[1] >= SENS_MIN, (name, "head tolerance cannot see a swapped coefficient chunk", head)


# ------------------------------------------------------------------------------------------------
# CPU: the harness against an emulation of the device's fp16 scheme
# ------------------------------------------------------------------------------------------------
class EmulatedDevice:
    """fp16 inputs and weights, fp32 convolutions, raw outputs rounded to fp16 where the library stores them in fp16 (first
    and last conv, edges above 64), InstanceNorm statistics of the fp32 raw output, fp16 layer outputs (the last conv's stays
    fp32: the head normalises it on load), fp32 head.  Nothing is normalised on load."""

    def __init__(self, net):
        self.net = rounded_copy(net, "fp16", torch.float32, "cpu")
        self.outs = []
        first, last = _first_conv(self.net), _last_conv(self.net)

        def on_layer(mod, inp, out):
            if isinstance(mod, O.ConvDropoutNormNonlin):
                y = mod.conv(inp[0])
                edge = max(y.shape[2:])
                yr = round_act(y, "fp16") if (mod is first or mod is last or edge > RAW32_MAX_EDGE) else y
                mean = y.double().mean(dim=(2, 3, 4), keepdim=True)
                var = y.double().var(dim=(2, 3, 4), unbiased=False, keepdim=True)
                a = (mod.instnorm.weight.double().view(1, -1, 1, 1, 1) / torch.sqrt(var + 1e-5)).float()
                b = mod.instnorm.bias.view(1, -1, 1, 1, 1) - a * mean.float()
                out = F.leaky_relu(a * yr + b, 1e-2)
                if mod is not last:
                    out = round_act(out, "fp16")
            else:
                out = round_act(out, "fp16")
            self.outs.append(out)
            return out

        for m in self.net.modules():
            if isinstance(m, (O.ConvDropoutNormNonlin, torch.nn.ConvTranspose3d)):
                m.register_forward_hook(on_layer)

    def forward_patches(self, x):
        self.outs = []
        with torch.no_grad():
            return torch.softmax(self.net(x.float()), 1)

    def layer_output(self, i, n=1):
        return self.outs[i][:n]

    def layer_norm_on_load(self, i):
        return 0

    def num_layers(self):
        return len(self.outs)


def test_tolerance_model_fits_an_fp16_emulation_and_sees_one_tap_errors():
    plans = small_plans()
    net = O.build_benchmark_network(0, plans)
    x = torch.randn(2, 1, 32, 32, 32, generator=torch.Generator().manual_seed(11))
    reports, head = layer_fp64_reports(net, EmulatedDevice(net), x, "fp16", "cpu")
    assert [r["kind"][:5] for r in reports].count("tconv") == 3 and len(reports) == 17
    check_reports("cpu-emulation", reports, head)
    # the mapping is by execution order: the transposed convs sit between the bottleneck and each decoder stage
    assert [i for i, r in enumerate(reports) if r["kind"].startswith("tconv")] == [8, 11, 14]


def test_tolerance_flags_an_emulated_device_that_drops_the_centre_tap():
    """The check works end to end: a device layer computed without its centre tap fails the bound."""
    plans = small_plans()
    net = O.build_benchmark_network(0, plans)
    broken = copy.deepcopy(net)
    with torch.no_grad():
        broken.conv_blocks_context[1].blocks[1].conv.weight[:, :, 1, 1, 1] = 0
    dev = EmulatedDevice(broken)
    x = torch.randn(1, 1, 32, 32, 32, generator=torch.Generator().manual_seed(12))
    reports, _ = layer_fp64_reports(net, dev, x, "fp16", "cpu")
    errs = [r["err"] for r in reports]
    assert errs[3] > SENS_MIN and max(errs[:3]) <= 1.0 and max(errs[4:]) <= 1.0, errs


def test_tolerance_flags_an_emulated_head_with_a_swapped_coefficient_chunk():
    """Eight classes: a device head that reads the last class's channels 0-3 where 4-7 belong fails the head bound,
    while every layer before it still passes."""
    plans = small_plans()
    plans["num_classes"] = 7
    net = O.build_benchmark_network(0, plans)
    broken = copy.deepcopy(net)
    with torch.no_grad():
        broken.seg_outputs[-1].weight.copy_(swap_last_class_chunks(broken.seg_outputs[-1].weight))
    x = torch.randn(1, 1, 32, 32, 32, generator=torch.Generator().manual_seed(13))
    reports, head = layer_fp64_reports(net, EmulatedDevice(broken), x, "fp16", "cpu")
    assert max(r["err"] for r in reports) <= 1.0
    assert head[0] > SENS_MIN, head
    _, head_ok = layer_fp64_reports(net, EmulatedDevice(net), x, "fp16", "cpu")
    assert head_ok[0] <= 1.0 and head_ok[1] >= SENS_MIN, head_ok


# ------------------------------------------------------------------------------------------------
# GPU: every configuration of DESIGN section 4's kernel paths
# ------------------------------------------------------------------------------------------------
def _bench_plans():
    import deepwmh_b200
    return deepwmh_b200.benchmark_plans()


_ANISO_A = dict(patch=(16, 64, 48), pools=((1, 2, 2), (2, 2, 2), (2, 2, 2)), kernels=[[1, 3, 3], [3, 3, 3], [3, 3, 3], [3, 3, 3]])
_ANISO_B = dict(patch=(8, 64, 64), pools=((1, 2, 2), (1, 2, 2), (2, 2, 2)), kernels=[[1, 3, 3], [1, 3, 3], [3, 3, 3], [3, 3, 3]])

# name: (plans factory, batch size, activation type, CUDA-core kernels forced)
CASES = {
    "small-n1": (lambda: small_plans(), 1, "fp16", False),
    "small-n2": (lambda: small_plans(), 2, "fp16", False),
    "small-n3": (lambda: small_plans(), 3, "fp16", False),
    "partial-64x48x40": (lambda: small_plans(patch=(64, 48, 40)), 2, "fp16", False),
    "aniso-16x64x48": (lambda: small_plans(**_ANISO_A), 2, "fp16", False),
    "aniso-8x64x64": (lambda: small_plans(**_ANISO_B), 2, "fp16", False),
    "base64-32x40x24": (lambda: small_plans(patch=(32, 40, 24), pools=((2, 2, 2),) * 2, base=64), 2, "fp16", False),
    "deep-64^3": (lambda: small_plans(patch=(64, 64, 64), pools=((2, 2, 2),) * 5), 2, "fp16", False),
    "nol32-72x88x44": (lambda: small_plans(patch=(72, 88, 44), pools=((2, 2, 2),) * 2), 2, "fp16", False),
    "nol64-72x88x44": (lambda: small_plans(patch=(72, 88, 44), pools=((2, 2, 2),) * 2, base=64), 2, "fp16", False),
    "nol32-72x80x40-n1": (lambda: small_plans(patch=(72, 80, 40), pools=((2, 2, 2),) * 2), 1, "fp16", False),
    "bench-128^3-n1": (_bench_plans, 1, "fp16", False),
    "bench-128^3-n3": (_bench_plans, 3, "fp16", False),
    "small-bf16": (lambda: small_plans(), 2, "bf16", False),
    "small-generic": (lambda: small_plans(), 2, "fp16", True),
    "partial-generic": (lambda: small_plans(patch=(64, 48, 40)), 2, "fp16", True),
    # the issue forms tests/test_conv_paths.py found unchecked by the cases above (its REQUIRED set; ADDED_FOR there
    # names the forms each of these reaches)
    "dstride-32x64x64-n3": (lambda: small_plans(patch=(32, 64, 64), pools=((2, 1, 1), (2, 2, 2), (2, 2, 2))), 3, "fp16", False),
    "k133stream-4x64x64": (lambda: small_plans(patch=(4, 64, 64), pools=((1, 2, 2),) * 4, kernels=[[1, 3, 3]] * 5), 2, "fp16", False),
    "nol32-72x80x40-n1-bf16": (lambda: small_plans(patch=(72, 80, 40), pools=((2, 2, 2),) * 2), 1, "bf16", False),
}

# The production batch: bench.py and predict_3D run max_batch = 32 forwards per launch, and the last batch of a tile range
# runs fewer on the same context.  name: (plans factory, batch size, max_batch, activation type, samples checked).  The
# device runs the whole batch of distinct patches; the float64 reference runs the listed samples only.
BATCH_CASES = {
    "bench-128^3-n32": (_bench_plans, 32, 32, "fp16", (0, 13, 31)),
    "bench-128^3-n17-of-32": (_bench_plans, 17, 32, "fp16", (0, 8, 16)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_every_layer_matches_fp64_on_its_own_inputs(case):
    import deepwmh_b200
    make_plans, n, act, generic = CASES[case]
    plans = make_plans()
    ps = tuple(int(i) for i in plans["plans_per_stage"][0]["patch_size"])
    net = O.build_benchmark_network(0, plans)
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, act_dtype=act, max_batch=n)
    tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
    nw = tr.network
    try:
        nw.set_force_generic(generic)
        kinds = [nw.layer_kernel_kind(i) for i in range(nw.num_layers())]
        if generic:
            assert not any(kinds), kinds
        else:
            assert sum(kinds) >= len(kinds) - 1, kinds      # every layer but possibly the first on tcgen05
        if case.startswith("nol"):
            assert any(nw.layer_norm_on_load(i) for i in range(nw.num_layers()))
        x = torch.randn(n, 1, *ps, generator=torch.Generator().manual_seed(7)).cuda()
        reports, head = layer_fp64_reports(net, nw, x, act)
        check_reports(case, reports, head)
    finally:
        nw.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(BATCH_CASES))
def test_every_layer_matches_fp64_at_the_production_batch(case):
    import deepwmh_b200
    make_plans, n, max_batch, act, samples = BATCH_CASES[case]
    plans = make_plans()
    ps = tuple(int(i) for i in plans["plans_per_stage"][0]["patch_size"])
    net = O.build_benchmark_network(0, plans)
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, act_dtype=act, max_batch=max_batch)
    tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
    nw = tr.network
    try:
        kinds = [nw.layer_kernel_kind(i) for i in range(nw.num_layers())]
        assert sum(kinds) >= len(kinds) - 1, kinds
        x = torch.randn(n, 1, *ps, generator=torch.Generator().manual_seed(7)).cuda()
        reports, head = layer_fp64_reports(net, nw, x, act, samples=samples)
        check_reports(case, reports, head)
    finally:
        nw.close()
