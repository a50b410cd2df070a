"""TEST INFRASTRUCTURE ONLY -- CPU restatement (numpy, fp64) of N4 bias-field correction as DeepWMH_predict runs it
(deepwmh/main/predict.py:117-126: `N4BiasFieldCorrection -d 3 -c [50x50x50x50,0.0] -s 2`, no mask, no weight image).

PARITY UNPINNED.  N4 lives in ITK / ANTs, neither of which is vendored or installed here.  The algorithm is restated
from its publications -- Tustison et al. 2010 (N4ITK), Sled et al. 1998 (N3 histogram sharpening), Lee, Wolberg & Shin
1997 (multilevel B-spline approximation) -- with the parameters DeepWMH passes and ANTs' defaults for the rest.  Details
of ITK's implementation that are recalled rather than checked against its source are marked [U]:
  * [U] voxels <= 0 take no part in the histogram or the fit (their log is undefined); no mask otherwise (ANTs without -x).
  * [U] itk::ShrinkImageFilter: output extent floor(N / s), no averaging, the voxel nearest each block's centre
        (index i * s + s // 2; the half-way case of an even s rounds up).
  * [U] histogram: 200 bins centred on min + n * slope, slope = (max - min) / 199, linear splatting into the two
        neighbouring bins; zero-padded to 512 = 2^(ceil(log2 200) + 1) points at offset floor((512 - 200) / 2) = 156.
  * [U] Wiener deconvolution with the circular Gaussian of FWHM 0.15 / slope bins (F[0] = 2 sqrt(ln 2 / pi) / FWHM,
        F[n] = F[512 - n] = F[0] exp(-4 ln 2 n^2 / FWHM^2)), G = conj(F^) / (|F^|^2 + 0.01); E[u | u^] as the ratio of
        the F-smoothed bin-centre-weighted and plain deconvolved histograms, 0 where the denominator is 0; linear lookup.
  * [U] B-spline fit: single-level Lee BSA of the residual with unit point weights, control lattices added level by
        level; refinement between levels by exact knot insertion (mesh doubling).
  * Parametric domain: the FULL-resolution index extent [0, N - 1] per axis is mapped to [0, mesh]; a shrunk point
        sits at its full-resolution index.  ANTs defines the domain from the image's physical extent; with mesh 1 on
        every axis this choice makes the result independent of voxel spacing.  This is the place ANTs may differ most.
Convergence threshold 0.0 (DeepWMH's): every iteration runs.
Only tests/ and tests/tools/ import this module.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np

BINS = 200
FWHM = 0.15
WIENER_NOISE = 0.01
PAD = 512
HIST_OFFSET = (PAD - BINS) // 2


def shrink_indices(n: int, s: int) -> np.ndarray:
    """Full-resolution indices of the floor(n / s) points itk::ShrinkImageFilter keeps along one axis [U]."""
    return np.arange(n // s, dtype=np.int64) * s + s // 2


def basis_matrix(t: np.ndarray, n_full: int, mesh: int) -> np.ndarray:
    """Dense cubic B-spline weights [len(t)][mesh + 3] of full-resolution indices t on the domain [0, n_full - 1] -> [0, mesh].
    Span k = floor(u) (k = mesh - 1 at u = mesh) weighs control points k .. k + 3."""
    t = np.asarray(t, dtype=np.int64)
    u = (t * mesh).astype(np.float64) / float(n_full - 1)
    k = np.minimum(np.floor(u).astype(np.int64), mesh - 1)
    x = u - k
    w = np.stack([(1 - x) ** 3 / 6, (3 * x ** 3 - 6 * x ** 2 + 4) / 6, (-3 * x ** 3 + 3 * x ** 2 + 3 * x + 1) / 6, x ** 3 / 6], 1)
    out = np.zeros((len(t), mesh + 3))
    for q in range(4):
        out[np.arange(len(t)), k + q] = w[:, q]
    return out


def evaluate(phi: np.ndarray, wx: np.ndarray, wy: np.ndarray, wz: np.ndarray) -> np.ndarray:
    """Field (Wx x Wy x Wz) phi on the grid of the three weight tables."""
    t = np.tensordot(wx, phi, axes=(1, 0))            # [i][b][c]
    t = np.tensordot(t, wy, axes=(1, 1))              # [i][c][j]
    t = np.tensordot(t, wz, axes=(1, 1))              # [i][j][k]
    return t


def contract(vol: np.ndarray, wx: np.ndarray, wy: np.ndarray, wz: np.ndarray) -> np.ndarray:
    """(Wx x Wy x Wz)^T vol -> control lattice [a][b][c]."""
    t = np.tensordot(vol, wz, axes=(2, 0))            # [i][j][c]
    t = np.tensordot(t, wy, axes=(1, 0))              # [i][c][b]
    t = np.tensordot(wx, t, axes=(0, 0))              # [a][c][b]
    return t.transpose(0, 2, 1)


def refine_matrix(mesh: int) -> np.ndarray:
    """Exact knot insertion of a uniform cubic B-spline, mesh -> 2 mesh: [2 mesh + 3][mesh + 3].  Coarse control point c
    (at u = c - 1) splits into fine points 2c - 3 .. 2c + 1 with weights (1, 4, 6, 4, 1) / 8; the fine points that fall
    outside the refined lattice have no support on the domain."""
    c_in, c_out = mesh + 3, 2 * mesh + 3
    r = np.zeros((c_out, c_in))
    for c in range(c_in):
        for e, w in zip(range(-2, 3), (1, 4, 6, 4, 1)):
            d = 2 * c - 1 + e
            if 0 <= d < c_out:
                r[d, c] = w / 8.0
    return r


def refine(phi: np.ndarray) -> np.ndarray:
    r = refine_matrix(phi.shape[0] - 3)
    return np.einsum("da,eb,fc,abc->def", r, r, r, phi, optimize=True)


def sharpen_table(hist: np.ndarray, bin_min: float, slope: float, fwhm: float = FWHM, noise: float = WIENER_NOISE) -> np.ndarray:
    """E[u | u^] at the BINS bin centres: Wiener deconvolution of the padded histogram with a Gaussian of FWHM fwhm (in
    the units of u), the FFT formulation ITK uses [U]."""
    v = np.zeros(PAD)
    v[HIST_OFFSET:HIST_OFFSET + BINS] = hist
    s_fwhm = fwhm / slope
    exp_f = 4.0 * np.log(2.0) / s_fwhm ** 2
    scale = 2.0 * np.sqrt(np.log(2.0) / np.pi) / s_fwhm
    f = np.zeros(PAD)
    f[0] = scale
    n = np.arange(1, PAD // 2 + 1)
    f[n] = scale * np.exp(-(n.astype(np.float64) ** 2) * exp_f)
    f[PAD - n] = f[n]
    ff = np.fft.fft(f)
    gf = np.conj(ff) / (np.conj(ff) * ff + noise)
    u = np.maximum(np.real(np.fft.ifft(np.fft.fft(v) * gf)), 0.0)
    centres = bin_min + (np.arange(PAD) - HIST_OFFSET) * slope
    num = np.real(np.fft.ifft(np.fft.fft(centres * u) * ff))[HIST_OFFSET:HIST_OFFSET + BINS]
    den = np.real(np.fft.ifft(np.fft.fft(u) * ff))[HIST_OFFSET:HIST_OFFSET + BINS]
    return np.where(den != 0, num / np.where(den != 0, den, 1.0), 0.0)


def sharpen(u: np.ndarray, fwhm: float = FWHM) -> np.ndarray:
    """Histogram-sharpened values of the samples u (1-D, fp64).  A constant u is returned unchanged."""
    lo, hi = float(u.min()), float(u.max())
    if not hi > lo:
        return u.copy()
    slope = (hi - lo) / (BINS - 1)
    cidx = (u - lo) / slope
    idx = np.minimum(np.floor(cidx).astype(np.int64), BINS - 1)
    off = np.where(idx == BINS - 1, 0.0, cidx - idx)
    hist = np.bincount(idx, 1.0 - off, BINS) + np.bincount(np.minimum(idx + 1, BINS - 1), off, BINS)
    e = sharpen_table(hist, lo, slope, fwhm)
    return np.where(idx < BINS - 1, e[idx] + (e[np.minimum(idx + 1, BINS - 1)] - e[idx]) * (cidx - idx), e[BINS - 1])


def n4(volume: np.ndarray, shrink: int = 2, iterations: Sequence[int] = (50, 50, 50, 50), return_log_field: bool = False):
    """N4 of an [X][Y][Z] volume: corrected = volume / exp(B), B the log bias field (fp64 throughout)."""
    img = np.asarray(volume, dtype=np.float64)
    dims = img.shape
    pts = [shrink_indices(n, shrink) for n in dims]
    if min(len(p) for p in pts) < 2:
        raise ValueError("shrink factor %d leaves fewer than 2 points on an axis of %s" % (shrink, dims))
    s = img[np.ix_(*pts)]
    valid = s > 0
    log_i = np.log(np.where(valid, s, 1.0))
    phi = np.zeros((4, 4, 4))
    for level, iters in enumerate(iterations):
        mesh = 2 ** level
        if level > 0:
            phi = refine(phi)
        w = [basis_matrix(p, n, mesh) for p, n in zip(pts, dims)]
        sw2 = [np.sum(x ** 2, 1) for x in w]
        inv_s = 1.0 / (sw2[0][:, None, None] * sw2[1][None, :, None] * sw2[2][None, None, :])
        omega = contract(valid.astype(np.float64), *[x ** 2 for x in w])
        w3 = [x ** 3 for x in w]
        for _ in range(iters):
            u = log_i - evaluate(phi, *w)
            r = np.zeros_like(u)
            r[valid] = u[valid] - sharpen(u[valid])
            delta = contract(r * inv_s, *w3)
            phi = phi + np.where(omega > 0, delta / np.where(omega > 0, omega, 1.0), 0.0)
    mesh = 2 ** (len(iterations) - 1)
    field = evaluate(phi, *[basis_matrix(np.arange(n), n, mesh) for n in dims])
    out = img / np.exp(field)
    return (out, field) if return_log_field else out


def phantom(shape: Tuple[int, int, int], seed: int = 0, amplitude: float = 0.2, noise: float = 0.03):
    """Seeded N4 test volume: three tissue classes of nested ellipsoids (intensities 250 / 520 / 800, multiplicative
    Gaussian noise of relative sd `noise`) in a zero background, multiplied by exp(f), f a random smooth field on a
    coarse cubic lattice (mesh 2) scaled to max |f| = amplitude.  Returns (image fp32, f fp64 [X][Y][Z], labels int8)."""
    rng = np.random.default_rng(seed)
    g = [np.linspace(-1.0, 1.0, n) for n in shape]
    x, y, z = np.meshgrid(*g, indexing="ij")
    c = rng.uniform(-0.05, 0.05, 3)
    r = np.sqrt(((x - c[0]) / 0.9) ** 2 + ((y - c[1]) / 0.85) ** 2 + ((z - c[2]) / 0.8) ** 2)
    labels = np.zeros(shape, np.int8)
    labels[r <= 1.0] = 1
    labels[r <= 0.75] = 2
    labels[r <= 0.45] = 3
    clean = np.choose(labels, [0.0, 250.0, 520.0, 800.0])
    clean = clean * (1.0 + noise * rng.standard_normal(shape))
    phi = rng.uniform(-1.0, 1.0, (5, 5, 5))
    f = evaluate(phi, *[basis_matrix(np.arange(n), n, 2) for n in shape])
    f = f - f.mean()
    f *= amplitude / np.abs(f).max()
    img = np.where(labels > 0, clean * np.exp(f), 0.0)
    return img.astype(np.float32), f, labels
