"""Stage-1 NLL anomaly map on the device (SURVEY.md section 8f-4).

Host-side mirror of the array functions the reference uses in `nll_analysis`
(deepwmh/analysis/lesion_analysis.py:115-181): same names, argument meaning and defaults as

    z_score, mean_std_grid, median_filter, median_3mm, group_mean, group_std,
    component_filtering                                                        deepwmh/analysis/image_ops.py
    nll                                                                        deepwmh/analysis/lesion_analysis.py:84-113

over the `dwmh_s1_*` entry points of include/deepwmh_b200.h.  Inputs may be numpy arrays or CUDA tensors [X, Y, Z];
results are fp32 CUDA tensors.  There is no CPU path: every function needs the library and a GPU.

`threshold_otsu` restates skimage's published 256-bin algorithm (skimage is not vendored by the reference; that piece is
`parity unpinned`).  Not built: the NIfTI / plot output of `nll_analysis`.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from ._lib import ptr, stream

Array = Union[np.ndarray, torch.Tensor]


def _dev(t: Array, device: int, copy: bool = False) -> torch.Tensor:
    """fp32 contiguous CUDA tensor (a fresh one when `copy`, so in-place kernels never touch the caller's data)."""
    if isinstance(t, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(t, dtype=np.float32)).to(f"cuda:{device}")
    out = t.to(device=f"cuda:{device}", dtype=torch.float32).contiguous()
    if copy and out.data_ptr() == t.data_ptr():
        out = out.clone()
    return out


def _i3(v: Sequence[int]):
    if len(v) != 3:
        raise ValueError("expected three values, got %r" % (v,))
    return (C.c_int32 * 3)(*[int(a) for a in v])


def _check3d(t: torch.Tensor, what: str):
    if t.dim() != 3:
        raise ValueError(f"{what} must be a 3-D volume, got shape {tuple(t.shape)}")


def z_score(data: Array, mask: Optional[Array] = None, fill_outside: bool = False, device: int = 0,
            return_stats: bool = False):
    """image_ops.py:172-179.  `fill_outside=True` also replaces the voxels outside the mask by the minimum inside it
    (lesion_analysis.py:150-151 / 160-161)."""
    lib = _lib.load()
    x = _dev(data, device, copy=True)
    m = _dev(mask, device) if mask is not None else None
    if m is not None and m.shape != x.shape:
        raise ValueError("z_score: mask shape %s != data shape %s" % (tuple(m.shape), tuple(x.shape)))
    ws = torch.empty(16, dtype=torch.float64, device=x.device)
    stats = (C.c_double * 3)() if return_stats else None
    with torch.cuda.device(x.device):
        _lib.check(lib.dwmh_s1_zscore(device, ptr(x), ptr(m), x.numel(), int(bool(fill_outside)), ptr(ws), stats, stream(device)))
    return (x, tuple(stats)) if return_stats else x


def z_score_batch_(volumes: Sequence[torch.Tensor], mask: Optional[Array] = None, fill_outside: bool = False) -> Sequence[torch.Tensor]:
    """z_score of up to 33 fp32 CUDA volumes sharing one mask, IN PLACE, in one pair of launches."""
    lib = _lib.load()
    if not volumes:
        return volumes
    dev = volumes[0].device
    for v in volumes:
        if v.device != dev or v.dtype != torch.float32 or not v.is_contiguous() or v.shape != volumes[0].shape:
            raise ValueError("z_score_batch_: volumes must be contiguous fp32 CUDA tensors of one shape on one device")
    m = _dev(mask, dev.index) if mask is not None else None
    if m is not None and m.shape != volumes[0].shape:
        raise ValueError("z_score_batch_: mask shape %s != data shape %s" % (tuple(m.shape), tuple(volumes[0].shape)))
    ws = torch.empty(8 * len(volumes), dtype=torch.float64, device=dev)
    ptrs = (C.c_void_p * len(volumes))(*[v.data_ptr() for v in volumes])
    with torch.cuda.device(dev):
        _lib.check(lib.dwmh_s1_zscore_batch(dev.index, ptrs, len(volumes), ptr(m), volumes[0].numel(), int(bool(fill_outside)),
                                            ptr(ws), stream(dev.index)))
    return volumes


def local_mean_align_(target: torch.Tensor, refs: Sequence[torch.Tensor], patch_size: Sequence[int], mask: Optional[Array] = None,
                      return_local_mean: bool = True) -> Optional[torch.Tensor]:
    """lesion_analysis.py:163-169 for a whole case in three launches: masked 50 mm local means of the target and of every
    reference, references aligned IN PLACE (x_i - x_i_local_mu + x_prime_local_mu).  -> x_prime_local_mu (or None)."""
    lib = _lib.load()
    dev = target.device
    _check3d(target, "local_mean_align_: target")
    for v in [target] + list(refs):
        if v.device != dev or v.dtype != torch.float32 or not v.is_contiguous() or v.shape != target.shape:
            raise ValueError("local_mean_align_: volumes must be contiguous fp32 CUDA tensors of one shape on one device")
    m = _dev(mask, dev.index) if mask is not None else None
    X, Y, Z = (int(v) for v in target.shape)
    ps = _i3(patch_size)
    nbytes = C.c_int64(0)
    _lib.check(lib.dwmh_s1_local_mean_align_workspace(X, Y, Z, ps, len(refs), C.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
    mu = torch.empty_like(target) if return_local_mean else None
    ptrs = (C.c_void_p * max(1, len(refs)))(*[r.data_ptr() for r in refs])
    with torch.cuda.device(dev):
        _lib.check(lib.dwmh_s1_local_mean_align(dev.index, ptr(target), ptrs, len(refs), ptr(m), X, Y, Z, ps, ptr(mu), ptr(ws),
                                                stream(dev.index)))
    return mu


def mean_std_grid(data: Array, patch_size: Sequence[int], order: int = 1, mask: Optional[Array] = None,
                  device: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """image_ops.py:56-170 (order 1, the value every call site in the reference uses)."""
    if order != 1:
        raise NotImplementedError("mean_std_grid: only order=1 (linear) is built; the reference never passes another order")
    lib = _lib.load()
    x = _dev(data, device)
    _check3d(x, "mean_std_grid: data")
    m = _dev(mask, device) if mask is not None else None
    if m is not None and m.shape != x.shape:
        raise ValueError("mean_std_grid: mask shape %s != data shape %s" % (tuple(m.shape), tuple(x.shape)))
    X, Y, Z = (int(v) for v in x.shape)
    ps = _i3(patch_size)
    nbytes = C.c_int64(0)
    _lib.check(lib.dwmh_s1_mean_std_grid_workspace(X, Y, Z, ps, C.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=x.device)
    mean, std = torch.empty_like(x), torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(lib.dwmh_s1_mean_std_grid(device, ptr(x), ptr(m), X, Y, Z, ps, ptr(mean), ptr(std), ptr(ws), stream(device)))
    return mean, std


def align_local_mean_(x: torch.Tensor, local_mu: torch.Tensor, target_local_mu: torch.Tensor) -> torch.Tensor:
    """lesion_analysis.py:166-169: x_i = x_i - x_i_local_mu + x_prime_local_mu, in place."""
    lib = _lib.load()
    device = x.device.index
    with torch.cuda.device(x.device):
        _lib.check(lib.dwmh_s1_align_local_mean(device, ptr(x), ptr(local_mu), ptr(target_local_mu), x.numel(), stream(device)))
    return x


def _side(side: Optional[str]) -> int:
    assert side in [None, "+", "-"]
    return {None: 0, "+": 1, "-": -1}[side]


def _group_nll(x: torch.Tensor, refs: Sequence[torch.Tensor], masks: Optional[Sequence[torch.Tensor]], min_std: float, side: int,
               mul_mask: Optional[torch.Tensor], want_an: bool, want_stats: bool):
    lib = _lib.load()
    device = x.device.index
    for r in list(refs) + list(masks or []):
        if r.shape != x.shape:
            raise ValueError("reference / mask shape %s != target shape %s" % (tuple(r.shape), tuple(x.shape)))
    if masks is not None and len(masks) != len(refs):
        raise ValueError("one mask per reference image is required")
    an = torch.empty_like(x) if want_an else None
    mu = torch.empty_like(x) if want_stats else None
    sg = torch.empty_like(x) if want_stats else None
    ptrs = (C.c_void_p * len(refs))(*[r.data_ptr() for r in refs])
    with torch.cuda.device(x.device):
        if masks is None:
            _lib.check(lib.dwmh_s1_group_nll(device, ptr(x), ptrs, len(refs), min_std, side, ptr(mul_mask), ptr(an), ptr(mu), ptr(sg),
                                             x.numel(), stream(device)))
        else:
            mptrs = (C.c_void_p * len(masks))(*[m.data_ptr() for m in masks])
            _lib.check(lib.dwmh_s1_group_nll_masked(device, ptr(x), ptrs, mptrs, len(refs), min_std, side, ptr(mul_mask), ptr(an),
                                                    ptr(mu), ptr(sg), x.numel(), stream(device)))
    return an, mu, sg


def nll(x_prime: Array, x_refs: Sequence[Array], min_std: Optional[float] = None, side: Optional[str] = None,
        return_all: bool = False, use_mask: bool = False, mul_mask: Optional[Array] = None, device: int = 0):
    """lesion_analysis.py:84-113.  `use_mask`: every reference counts only where it exceeds its own Otsu threshold (:87-92).
    `mul_mask` (not in the reference signature) fuses the `anomaly * m_valid_score` that follows every call (:175, :184)."""
    x = _dev(x_prime, device)
    refs = [_dev(r, device) for r in x_refs]
    if not refs:
        raise ValueError("nll: no reference images")
    masks = [threshold_mask(r, threshold_otsu(r, device=device), device=device) for r in refs] if use_mask else None
    mm = _dev(mul_mask, device) if mul_mask is not None else None
    an, mu, sg = _group_nll(x, refs, masks, -1.0 if min_std is None else float(min_std), _side(side), mm, True, return_all)
    return (an, mu, sg) if return_all else an


def group_mean(data_list: Sequence[Array], masks: Optional[Sequence[Array]] = None, device: int = 0) -> torch.Tensor:
    """image_ops.py:216-231 (NaN where every image is masked out)."""
    return _group(data_list, masks, device)[0]


def group_std(data_list: Sequence[Array], masks: Optional[Sequence[Array]] = None, device: int = 0) -> torch.Tensor:
    """image_ops.py:199-214: population std."""
    return _group(data_list, masks, device)[1]


def _group(data_list, masks, device):
    refs = [_dev(r, device) for r in data_list]
    ms = [_dev(m, device) for m in masks] if masks is not None else None
    # min_std = 0: sigma is returned unmodified
    _, mu, sg = _group_nll(refs[0], refs, ms, 0.0, 0, None, False, True)
    return mu, sg


def median_filter(data: Array, kernel_size: Sequence[int], device: int = 0) -> torch.Tensor:
    """image_ops.py:181-183: scipy.ndimage.median_filter(size=kernel_size, mode='constant', cval=0), 3-D."""
    lib = _lib.load()
    x = _dev(data, device)
    _check3d(x, "median_filter: data")
    out = torch.empty_like(x)
    X, Y, Z = (int(v) for v in x.shape)
    with torch.cuda.device(x.device):
        _lib.check(lib.dwmh_s1_median_filter(device, ptr(x), ptr(out), X, Y, Z, _i3(kernel_size), stream(device)))
    return out


def median_kernel_size(physical_voxel_size: Sequence[float]) -> List[int]:
    """The kernel rule of median_3mm (image_ops.py:378-421): int(3 mm / voxel) per axis, at least 3; thick-slice data
    (max / min > 4) is filtered slice by slice, i.e. with size 1 along the thick axis."""
    vs = [float(v) for v in physical_voxel_size]
    ks = [max(3, int(3.0 / v)) for v in vs]
    if max(vs) / min(vs) > 4.0:
        ks[int(np.argmax(vs))] = 1
    return ks


def median_3mm(data: Array, physical_voxel_size: Sequence[float], device: int = 0) -> torch.Tensor:
    return median_filter(data, median_kernel_size(physical_voxel_size), device=device)


def component_filtering(mask: Array, voxel_size: Sequence[float], return_type: str = "float32", erosion: bool = True,
                        device: int = 0) -> torch.Tensor:
    """image_ops.py:253-306 ("quickly refines the calculated brain mask"); `erosion` is accepted and, as in the reference,
    ignored (the slices are always eroded)."""
    if return_type != "float32":
        raise NotImplementedError("component_filtering: only return_type='float32' is built")
    lib = _lib.load()
    m = _dev(mask, device)
    _check3d(m, "component_filtering: mask")
    X, Y, Z = (int(v) for v in m.shape)
    if len(voxel_size) != 3:
        raise ValueError("component_filtering: voxel_size needs three values")
    vs = (C.c_double * 3)(*[float(v) for v in voxel_size])
    nbytes = C.c_int64(0)
    _lib.check(lib.dwmh_s1_component_filtering_workspace(X, Y, Z, C.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=m.device)
    out = torch.empty_like(m)
    with torch.cuda.device(m.device):
        _lib.check(lib.dwmh_s1_component_filtering(device, ptr(m), X, Y, Z, vs, ptr(out), ptr(ws), stream(device)))
    return out


def minmax(data: Array, mask: Optional[Array] = None, device: int = 0) -> Tuple[float, float]:
    lib = _lib.load()
    x = _dev(data, device)
    m = _dev(mask, device) if mask is not None else None
    ws = torch.empty(2, dtype=torch.int32, device=x.device)
    out = (C.c_float * 2)()
    with torch.cuda.device(x.device):
        _lib.check(lib.dwmh_s1_minmax(device, ptr(x), ptr(m), x.numel(), ptr(ws), out, stream(device)))
    return float(out[0]), float(out[1])


def histogram(data: Array, bin_edges: np.ndarray, mask: Optional[Array] = None, fill_value: Optional[float] = None,
              device: int = 0) -> np.ndarray:
    """numpy.histogram(values, bins=bin_edges) for equal-width edges; values = data[mask > 0.5], or
    np.where(mask < 0.5, fill_value, data) when fill_value is given.  -> int64 counts on the host."""
    lib = _lib.load()
    x = _dev(data, device)
    m = _dev(mask, device) if mask is not None else None
    edges = torch.from_numpy(np.ascontiguousarray(bin_edges, dtype=np.float64)).to(x.device)
    nbins = int(edges.numel()) - 1
    counts = torch.empty(nbins, dtype=torch.int64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.dwmh_s1_histogram(device, ptr(x), ptr(m), x.numel(), int(fill_value is not None),
                                         float(fill_value if fill_value is not None else 0.0), ptr(edges), nbins, ptr(counts), stream(device)))
    return counts.cpu().numpy()


def _otsu_from_histogram(counts: np.ndarray, bin_edges: np.ndarray) -> float:
    """The scan of skimage.filters.threshold_otsu: maximise the between-class variance over the 255 cut points."""
    counts = counts.astype(np.float64)
    centers = (bin_edges[:-1] + bin_edges[1:]) / 2.0
    w1 = np.cumsum(counts)
    w2 = np.cumsum(counts[::-1])[::-1]
    with np.errstate(divide="ignore", invalid="ignore"):
        m1 = np.cumsum(counts * centers) / w1
        m2 = (np.cumsum((counts * centers)[::-1]) / w2[::-1])[::-1]
    var12 = w1[:-1] * w2[1:] * (m1[:-1] - m2[1:]) ** 2
    return float(centers[int(np.argmax(var12))])


def threshold_otsu(image: Array, nbins: int = 256, mask: Optional[Array] = None, fill_value: Optional[float] = None,
                   device: int = 0) -> float:
    """skimage.filters.threshold_otsu(values), values = image (mask None), image[mask > 0.5] (`otsu_thresholding`,
    image_ops.py:308-323) or np.where(mask < 0.5, fill_value, image) (lesion_analysis.py:145)."""
    x = _dev(image, device)
    m = _dev(mask, device) if mask is not None else None
    lo, hi = minmax(x, m, device)
    if m is not None and fill_value is not None:
        lo, hi = min(lo, float(np.float32(fill_value))), max(hi, float(np.float32(fill_value)))
    if lo == hi:
        return lo                                                     # a single intensity: skimage returns it
    edges = np.linspace(lo, hi, nbins + 1)
    return _otsu_from_histogram(histogram(x, edges, m, fill_value, device), edges)


def otsu_thresholding(image: Array, mask: Optional[Array] = None, device: int = 0) -> Optional[float]:
    """image_ops.py:308-323."""
    if mask is not None and float(_dev(mask, device).gt(0.5).sum().item()) < 1:
        return None
    return threshold_otsu(image, mask=mask, device=device)


def threshold_mask(data: Array, threshold: float, mul_mask: Optional[Array] = None, device: int = 0) -> torch.Tensor:
    """np.where(data > threshold, 1, 0) [* mul_mask] as fp32."""
    lib = _lib.load()
    x = _dev(data, device)
    mm = _dev(mul_mask, device) if mul_mask is not None else None
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(lib.dwmh_s1_threshold_mask(device, ptr(x), float(threshold), ptr(mm), ptr(out), x.numel(), stream(device)))
    return out


def valid_score_mask(x_prime_raw: Array, m_rough_brain: Array, apply_otsu: bool = True, device: int = 0):
    """lesion_analysis.py:142-148: z-score the target over the rough brain mask, Otsu-threshold it (voxels outside the
    brain set to the volume minimum), m_valid_score = m_rough_brain * m_otsu.  -> (x_prime z-scored, m_valid_score)."""
    brain = _dev(m_rough_brain, device)
    xp = z_score(x_prime_raw, brain, device=device)
    if not apply_otsu:
        return xp, brain.clone()
    lo, _ = minmax(xp, None, device)
    thr = threshold_otsu(xp, mask=brain, fill_value=lo, device=device)
    return xp, threshold_mask(xp, thr, brain, device)


def image_patch_size(physical_voxel_size: Sequence[float], physical_patch_size=(50, 50, 50)) -> List[int]:
    """lesion_analysis.py:124-131: the 50 mm local-mean patch in voxels."""
    return [int(np.ceil(p / v)) for p, v in zip(physical_patch_size, physical_voxel_size)]


def nll_anomaly_map(x_prime: Array, x_refs: Sequence[Array], m_rough_brain: Array, m_valid_score: Array,
                    physical_voxel_size: Sequence[float] = (1.0, 1.0, 1.0), intensity_prior: Optional[str] = None,
                    mean_correction: bool = True, min_std: float = 0.03, image_patch: Optional[Sequence[int]] = None,
                    with_reference_scores: bool = False, apply_component_filtering: bool = False, device: int = 0) -> dict:
    """The array part of `nll_analysis` (lesion_analysis.py:142-186) from raw registered volumes and the two masks:
    z-score over the rough brain mask + tissue-min fill (target and every reference), 50 mm local-mean alignment of the
    references to the target, voxelwise Gaussian NLL with sigma floored at `min_std`, masked by the valid-score mask.
    -> dict of fp32 CUDA tensors: normalized_input, local_mean (masked as at :170), anomaly, mean, std
       [+ reference_anomalies, :179-185]."""
    assert intensity_prior in [None, "+", "-"], 'Unknown intensity prior "%s".' % str(intensity_prior)
    patch = list(image_patch) if image_patch is not None else image_patch_size(physical_voxel_size)
    brain = _dev(m_rough_brain, device)
    valid = _dev(m_valid_score, device)
    # one device copy per volume, then the whole case per launch: z-score + tissue-min fill of the k + 1 volumes (2 launches),
    # local means + alignment (3 launches), NLL (1 launch)
    xp = _dev(x_prime, device, copy=True)
    refs = [_dev(r, device, copy=True) for r in x_refs]
    z_score_batch_([xp] + refs, brain, fill_outside=True)
    mu_p = local_mean_align_(xp, refs if mean_correction else [], patch, mask=valid)
    an, mean, std = nll(xp, refs, min_std=min_std, side=intensity_prior, return_all=True, mul_mask=valid, device=device)
    if apply_component_filtering:                                    # lesion_analysis.py:176 (the target's score only)
        an = an * component_filtering(valid, physical_voxel_size, device=device)
    out = {"normalized_input": xp, "local_mean": mu_p * valid, "anomaly": an, "mean": mean, "std": std}
    if with_reference_scores:
        out["reference_anomalies"] = [nll(r, refs, min_std=min_std, side=intensity_prior, mul_mask=valid, device=device) for r in refs]
    return out


def masked_sums(volumes: Sequence[torch.Tensor], mask: Optional[Array] = None, positive_only: bool = False) -> np.ndarray:
    """{sum, sum of squares, count} per volume over mask > 0.5 (and value > 0), one launch -> float64 [nvol, 3] on the host."""
    lib = _lib.load()
    dev = volumes[0].device
    m = _dev(mask, dev.index) if mask is not None else None
    ws = torch.empty(8 * len(volumes), dtype=torch.float64, device=dev)
    out = (C.c_double * (3 * len(volumes)))()
    ptrs = (C.c_void_p * len(volumes))(*[v.data_ptr() for v in volumes])
    with torch.cuda.device(dev):
        _lib.check(lib.dwmh_s1_masked_sums(dev.index, ptrs, len(volumes), ptr(m), volumes[0].numel(), int(bool(positive_only)), ptr(ws),
                                           out, stream(dev.index)))
    return np.array(out, dtype=np.float64).reshape(len(volumes), 3)


def hist_curve(data: Array, bins: np.ndarray, log_y: bool = False, mask: Optional[Array] = None, device: int = 0):
    """lesion_analysis.py:40-50 (equal-width `bins` edges)."""
    hist = histogram(data, bins, mask=mask, device=device).astype(np.int64)
    bins = np.asarray(bins, np.float64)
    centers = (bins[:-1] + bins[1:]) / 2
    if log_y:
        hist = np.where(hist == 0, 0.001, hist)
        hist = np.log10(hist)
        hist = np.where(hist < 0, 0, hist)
    return centers, hist


def histogram_analysis(a_prime: Array, a_refs: Sequence[Array], bins: Optional[np.ndarray] = None, mask: Optional[Array] = None, device: int = 0):
    """lesion_analysis.py:52-82: log-histogram curves of the target's anomaly score and of every reference's; default bins =
    400 bins of width (mean over references of the mean positive masked score) / 4."""
    if not isinstance(a_refs, (list, tuple)):
        a_refs = [a_refs]
    refs = [_dev(r, device) for r in a_refs]
    if bins is None:
        assert mask is not None, 'must provide mask when "bins" is None.'
        sums = masked_sums(refs, mask, positive_only=True)
        ref_means = sums[:, 0] / sums[:, 2]
        bin_width = ref_means.mean() / 4
        num_bins = 400
        bins = np.linspace(0.0, 0.0 + num_bins * bin_width, num=num_bins + 1)
    x, y = hist_curve(a_prime, bins, log_y=True, device=device)
    rs = [hist_curve(r, bins, log_y=True, device=device)[1] for r in refs]
    r = np.zeros_like(x)
    for r0 in rs:
        r = r + r0
    return x, y, r / len(rs), rs


def anomaly_threshold_from_curves(curve_x: np.ndarray, curve_rs: Sequence[np.ndarray]) -> float:
    """lesion_analysis.py:194-207: per reference, the right-most histogram bin whose log-count exceeds 0.01; the initial
    segmentation threshold is the median of those positions."""
    zero_crossings = []
    for rs in curve_rs:
        for j in range(len(rs) - 1, 0, -1):
            if rs[j] > 0.01:
                zero_crossings.append(curve_x[j])
                break
    return float(np.median(np.sort(zero_crossings)))


def label_vote(labels: Sequence[Array], device: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """average_contiguous_labels (image_ops.py:23-38) and the tissue majority mask (lesion_analysis.py:238-242)."""
    lib = _lib.load()
    ls = [_dev(l, device) for l in labels]
    num = 1 + max(int(minmax(l, None, device)[1]) for l in ls)
    avg, tissue = torch.empty_like(ls[0]), torch.empty_like(ls[0])
    ptrs = (C.c_void_p * len(ls))(*[l.data_ptr() for l in ls])
    with torch.cuda.device(ls[0].device):
        _lib.check(lib.dwmh_s1_label_vote(device, ptrs, len(ls), num, ptr(avg), ptr(tissue), avg.numel(), stream(device)))
    return avg, tissue


def average_contiguous_labels(labels: Sequence[Array], device: int = 0) -> torch.Tensor:
    return label_vote(labels, device)[0]


def apply_priors_(anomaly: torch.Tensor, averaged_label: torch.Tensor, tissue_majority: Optional[torch.Tensor] = None,
                  anomaly_median: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Stage 1 (no median given): anomaly *= (averaged_label > 0.5).  Stage 2: cerebellum / brainstem voxels take the
    median-filtered score, everything is masked by the tissue majority vote.  In place."""
    lib = _lib.load()
    dev = anomaly.device
    with torch.cuda.device(dev):
        _lib.check(lib.dwmh_s1_apply_priors(dev.index, ptr(anomaly), ptr(anomaly_median), ptr(averaged_label), ptr(tissue_majority),
                                            1 if anomaly_median is None else 2, anomaly.numel(), stream(dev.index)))
    return anomaly


def nll_analysis_arrays(x: Array, x_refs: Sequence[Array], ref_label1: Sequence[Array], ref_label2: Sequence[Array],
                        physical_voxel_size: Sequence[float], apply_otsu: bool = True, intensity_prior: Optional[str] = None,
                        mean_correction: bool = True, device: int = 0):
    """`nll_analysis` (lesion_analysis.py:115-281) on arrays instead of NIfTI paths: x = case_info['x'], x_refs = ['r'],
    ref_label1 = ['m'] (brain masks of the references), ref_label2 = ['y'] (tissue labels 0..3).
    -> (anomaly, m_valid_score, curve_x, curve_y, curve_r, anomaly_threshold) as the reference returns them (volumes as fp32
    CUDA tensors), plus a dict with normalized_input / local_mean / mean / std / averaged_label / rough_brain."""
    assert intensity_prior in [None, "+", "-"], 'Unknown intensity prior "%s".' % str(intensity_prior)
    vox = [float(v) for v in physical_voxel_size]
    patch = image_patch_size(vox)
    m_i = [threshold_mask(l, 0.5, device=device) for l in ref_label1]
    m_rough_brain = threshold_mask(group_mean(m_i, device=device), 0.5, device=device)
    _, m_valid = valid_score_mask(x, m_rough_brain, apply_otsu=apply_otsu, device=device)
    r = nll_anomaly_map(x, x_refs, m_rough_brain, m_valid, vox, intensity_prior=intensity_prior, mean_correction=mean_correction,
                        min_std=0.03, image_patch=patch, with_reference_scores=True, apply_component_filtering=True, device=device)
    anomaly = r["anomaly"]
    curve_x, curve_y, curve_r, curve_rs = histogram_analysis(anomaly, r["reference_anomalies"], mask=m_valid, device=device)
    thr = anomaly_threshold_from_curves(curve_x, curve_rs)
    averaged_label, tissue = label_vote(ref_label2, device=device)
    apply_priors_(anomaly, averaged_label)
    apply_priors_(anomaly, averaged_label, tissue, median_3mm(anomaly, vox, device=device))
    extras = {"normalized_input": r["normalized_input"], "local_mean": r["local_mean"], "mean": r["mean"], "std": r["std"],
              "averaged_label": averaged_label, "rough_brain": m_rough_brain, "curve_rs": curve_rs}
    return anomaly, m_valid, curve_x, curve_y, curve_r, thr, extras
