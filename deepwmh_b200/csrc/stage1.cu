// SURVEY.md section 8f-4: nll_analysis of deepwmh/analysis/lesion_analysis.py:115-281 (the stage-1 NLL anomaly map) on the device.
// Voxel-parallel, HBM-bound kernels; fp32 storage, fp64 per-voxel arithmetic (the reference works in float64 once a
// volume has been z-scored).  Context-free entry points (no network involved): `device` + caller-owned buffers.
//
//   dwmh_s1_zscore[_batch]        z_score (image_ops.py:172-179) [+ tissue-min fill, lesion_analysis.py:150-151,160-161]
//   dwmh_s1_mean_std_grid         mean_std_grid, order 1 (image_ops.py:56-170)
//   dwmh_s1_local_mean_align      local means of a whole case + x_i - x_i_local_mu + x_prime_local_mu (lesion_analysis.py:163-169)
//   dwmh_s1_align_local_mean      the alignment alone, from materialised local means
//   dwmh_s1_group_nll[_masked]    group_mean / group_std / nll (image_ops.py:197-231, lesion_analysis.py:84-113)
//   dwmh_s1_median_filter         median_filter(mode='constant', cval=0) behind median_3mm (image_ops.py:181-183,378-421)
//   dwmh_s1_component_filtering   component_filtering (image_ops.py:253-306)
//   dwmh_s1_minmax / _histogram / _threshold_mask   Otsu mask (lesion_analysis.py:142-148) and hist_curve (:40-50)
//   dwmh_s1_masked_sums           bin width of histogram_analysis (:52-82)
//   dwmh_s1_label_vote / _apply_priors   average_contiguous_labels (image_ops.py:23-38) and the tissue priors (:213-243)
#include "../../include/deepwmh_b200.h"

#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>

#include "host.cuh"
#include "common.cuh"
#include "kernels_ccl.cuh"

using dwmh::fail;
using dwmh::sm_count;

namespace {

using dwmh::warp_sum_d;

// Batched launches: blockIdx.y selects one of up to S1_MAX_VOLS volumes (the target + its registered references).
constexpr int S1_MAX_REFS = 32;
constexpr int S1_MAX_VOLS = S1_MAX_REFS + 1;
struct VolPtrs { float* p[S1_MAX_VOLS]; };
constexpr int ZS_SLOT = 8;          // doubles per volume in the z-score workspace: {sum, sumsq, count, -, min (int), ...}

// order-preserving float <-> signed int (atomicMin on floats)
__device__ __forceinline__ int f2ord(float f) { const int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

// ---------------------------------------------------------------------------------------------------------------
// z_score.  ws: double[4] = {sum, sumsq, count, -} + int min (ordered) at byte 32.  Pass 1 reads x (+mask), pass 2
// reads x (+mask) and writes x: 12 B/voxel (+8 with a mask).
// ---------------------------------------------------------------------------------------------------------------
template <bool VEC>
__global__ void __launch_bounds__(256) s1_stats_kernel(VolPtrs vols, const float* __restrict__ mask,
                                                       int64_t n, double* __restrict__ ws, int positive_only = 0) {
  const float* __restrict__ x = vols.p[blockIdx.y];
  double* acc = ws + (size_t)blockIdx.y * ZS_SLOT;
  int* minord = reinterpret_cast<int*>(acc + 4);
  double s = 0.0, ss = 0.0, cnt = 0.0;
  int mn = 0x7fffffff;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n4 = VEC ? n >> 2 : 0;
  for (int64_t i = tid; i < n4; i += stride) {
    const float4 v = dwmh::ld_stream_f4(reinterpret_cast<const float4*>(x) + i);
    float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
    if (mask) m = dwmh::ld_stream_f4(reinterpret_cast<const float4*>(mask) + i);
    const float vv[4] = {v.x, v.y, v.z, v.w}, mm[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (mm[j] > 0.5f && (!positive_only || vv[j] > 0.f)) { s += vv[j]; ss += (double)vv[j] * vv[j]; cnt += 1.0; mn = min(mn, f2ord(vv[j])); }
  }
  for (int64_t i = (n4 << 2) + tid; i < n; i += stride) {
    const float v = x[i];
    if ((!mask || mask[i] > 0.5f) && (!positive_only || v > 0.f)) { s += v; ss += (double)v * v; cnt += 1.0; mn = min(mn, f2ord(v)); }
  }
  s = warp_sum_d(s); ss = warp_sum_d(ss); cnt = warp_sum_d(cnt);
  mn = __reduce_min_sync(0xffffffffu, mn);
  __shared__ double sh[3][8];
  __shared__ int shm[8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = s; sh[1][w] = ss; sh[2][w] = cnt; shm[w] = mn; }
  __syncthreads();
  if (w == 0) {
    s = l < 8 ? sh[0][l] : 0.0; ss = l < 8 ? sh[1][l] : 0.0; cnt = l < 8 ? sh[2][l] : 0.0; mn = l < 8 ? shm[l] : 0x7fffffff;
    s = warp_sum_d(s); ss = warp_sum_d(ss); cnt = warp_sum_d(cnt); mn = __reduce_min_sync(0xffffffffu, mn);
    if (l == 0) { atomicAdd(acc + 0, s); atomicAdd(acc + 1, ss); atomicAdd(acc + 2, cnt); atomicMin(minord, mn); }
  }
}

template <bool VEC>
__global__ void __launch_bounds__(256) s1_zscore_apply_kernel(VolPtrs vols, const float* __restrict__ mask, int64_t n,
                                                              const double* __restrict__ ws, int fill_outside) {
  float* __restrict__ x = vols.p[blockIdx.y];
  const double* acc = ws + (size_t)blockIdx.y * ZS_SLOT;
  const int* minord = reinterpret_cast<const int*>(acc + 4);
  const double cnt = acc[2] > 0.0 ? acc[2] : 1.0;
  const double mean = acc[0] / cnt;
  double var = acc[1] / cnt - mean * mean;
  var = var > 0.0 ? var : 0.0;
  const double sd = fmax(sqrt(var), 0.00001);                       // np.max([std, 1e-5])
  const float fill = (float)(((double)ord2f(*minord) - mean) / sd);   // z-scoring is monotone: min(z) = z(min)
  const bool do_fill = fill_outside && mask;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n4 = VEC ? n >> 2 : 0;
  for (int64_t i = tid; i < n4; i += stride) {
    float4 v = reinterpret_cast<const float4*>(x)[i];
    float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
    if (do_fill) m = dwmh::ld_stream_f4(reinterpret_cast<const float4*>(mask) + i);
    v.x = m.x >= 0.5f ? (float)(((double)v.x - mean) / sd) : fill;    // np.where(m < 0.5, tissue_min, x)
    v.y = m.y >= 0.5f ? (float)(((double)v.y - mean) / sd) : fill;
    v.z = m.z >= 0.5f ? (float)(((double)v.z - mean) / sd) : fill;
    v.w = m.w >= 0.5f ? (float)(((double)v.w - mean) / sd) : fill;
    reinterpret_cast<float4*>(x)[i] = v;
  }
  for (int64_t i = (n4 << 2) + tid; i < n; i += stride) {
    const float z = (float)(((double)x[i] - mean) / sd);
    x[i] = (do_fill && !(mask[i] >= 0.5f)) ? fill : z;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// mean_std_grid.  The blocks of the reference are patch-sized and half-overlapping, i.e. every block is the union of
// (up to) 2x2x2 step-sized cells: one CTA reduces one cell to {sum, sumsq, count} (the volume is read exactly once),
// a tiny kernel combines the cells into the zero-bordered mean / std grids, and the zoom kernel evaluates scipy's
// order-1 `zoom` of those grids at the voxels that survive the reference's cropping.
// ---------------------------------------------------------------------------------------------------------------
struct GridGeom {
  int X, Y, Z;          // data shape
  int st[3];            // step = patch / 2 (patch rounded up to even)
  int pad[3];           // padded shape (multiple of the patch)
  int g[3];             // cells per axis = pad / st = grid shape
  double scale[3];      // scipy zoom coordinate scale (in - 1) / (out - 1) of the bordered grid
};

// One CTA per (cell-x, cell-y, x-plane): thread t owns the z coordinates t, t + 256, ..., so every iteration
// reads one contiguous z-row of the volume (coalesced, 8 rows in flight) and a thread's running sums belong to ONE
// z-cell; the per-z sums are then folded into the z-cells through shared memory and added to `cells`
// (zeroed by the host) with a handful of fp64 atomics per CTA.
constexpr int CS_SLAB = 5;          // x-planes per CTA
__global__ void __launch_bounds__(256) s1_cell_sums_kernel(VolPtrs vols, const float* __restrict__ mask,
                                                           GridGeom q, int slabs, double* __restrict__ cells_all) {
  extern __shared__ double zs[];    // [3][min(Z, chunk)] per-z sums of the current z chunk
  const float* __restrict__ x = vols.p[blockIdx.y];
  double* cells = cells_all + (size_t)blockIdx.y * q.g[0] * q.g[1] * q.g[2] * 3;
  const int slab = blockIdx.x % slabs, cy = (blockIdx.x / slabs) % q.g[1], cx = blockIdx.x / (slabs * q.g[1]);
  const int x0 = cx * q.st[0] + slab * CS_SLAB, x1 = min(min(x0 + CS_SLAB, (cx + 1) * q.st[0]), q.X);
  const int y0 = cy * q.st[1], y1 = min(y0 + q.st[1], q.Y);
  const int T = blockDim.x;
  for (int zb = 0; zb < q.Z; zb += T) {
    const int z = zb + threadIdx.x;
    double s = 0.0, ss = 0.0, cnt = 0.0;
    if (z < q.Z)
      for (int xi = x0; xi < x1; ++xi) {
        const float* px = x + ((int64_t)xi * q.Y + y0) * q.Z + z;
        const float* pm = mask ? mask + ((int64_t)xi * q.Y + y0) * q.Z + z : nullptr;
#pragma unroll 8
        for (int yi = 0; yi < y1 - y0; ++yi) {
          const float v = __ldg(px + (int64_t)yi * q.Z);
          const bool m = !pm || __ldg(pm + (int64_t)yi * q.Z) > 0.5f;
          if (m) { s += v; ss += (double)v * v; cnt += 1.0; }
        }
      }
    zs[threadIdx.x] = s; zs[T + threadIdx.x] = ss; zs[2 * T + threadIdx.x] = cnt;
    __syncthreads();
    // fold the z coordinates of this chunk into their cells: one thread per (cell, quantity), a short sequential sum
    const int c_lo = zb / q.st[2], c_hi = min((min(zb + T, q.Z) - 1) / q.st[2], q.g[2] - 1);
    for (int i = threadIdx.x; i < 3 * (c_hi - c_lo + 1); i += T) {
      const int cz = c_lo + i / 3, w = i % 3;
      const int z_lo = max(cz * q.st[2], zb), z_hi = min(min((cz + 1) * q.st[2], zb + T), q.Z);
      double acc = 0.0;
      for (int zz = z_lo; zz < z_hi; ++zz) acc += zs[w * T + (zz - zb)];
      if (acc != 0.0) atomicAdd(cells + ((size_t)(cx * q.g[1] + cy) * q.g[2] + cz) * 3 + w, acc);
    }
    __syncthreads();
  }
}

// grids: [g0+2][g1+2][g2+2] doubles, borders zero (memset by the host)
__global__ void s1_grid_stats_kernel(const double* __restrict__ cells_all, GridGeom q, int masked,
                                     double* __restrict__ mean_grids, double* __restrict__ std_grids, size_t grid_stride) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= q.g[0] * q.g[1] * q.g[2]) return;
  const double* cells = cells_all + (size_t)blockIdx.y * q.g[0] * q.g[1] * q.g[2] * 3;
  double* mean_grid = mean_grids + blockIdx.y * grid_stride;
  double* std_grid = std_grids + blockIdx.y * grid_stride;
  const int k = t % q.g[2], j = (t / q.g[2]) % q.g[1], i = t / (q.g[2] * q.g[1]);
  double s = 0.0, ss = 0.0, cnt = 0.0;
  for (int a = i; a < min(i + 2, q.g[0]); ++a)                       // the last block is clipped by the padded shape
    for (int b = j; b < min(j + 2, q.g[1]); ++b)
      for (int c = k; c < min(k + 2, q.g[2]); ++c) {
        const double* p = cells + ((size_t)(a * q.g[1] + b) * q.g[2] + c) * 3;
        s += p[0]; ss += p[1]; cnt += p[2];
      }
  double mu, sd;
  if (masked) {
    if (cnt > 0.0) { mu = s / cnt; const double v = ss / cnt - mu * mu; sd = sqrt(v > 0.0 ? v : 0.0); }
    else { mu = 0.0; sd = 0.00001; }
  } else {                                                           // zero padding counts as data
    const double nb = (double)(min(i + 2, q.g[0]) - i) * q.st[0] * (double)(min(j + 2, q.g[1]) - j) * q.st[1] *
                      (double)(min(k + 2, q.g[2]) - k) * q.st[2];
    mu = s / nb; const double v = ss / nb - mu * mu; sd = fmax(sqrt(v > 0.0 ? v : 0.0), 0.00001);
  }
  const size_t o = ((size_t)(i + 1) * (q.g[1] + 2) + (j + 1)) * (q.g[2] + 2) + (k + 1);
  mean_grid[o] = mu; std_grid[o] = sd;
}

// scipy.ndimage.zoom(grid, step, order=1): output index o <-> input coordinate o * (in - 1) / (out - 1)
__device__ __forceinline__ void zoom_coord(int v, int st, int g, double scale, int& i0, double& f) {
  const double c = (double)(v + st / 2) * scale;
  i0 = (int)floor(c);
  f = c - (double)i0;
  if (i0 >= g + 1) { i0 = g; f = 1.0; }
}

// Linear zoom is separable: for one (x, y) row the four x/y corner rows of the coarse grid collapse into ONE z-profile
// prof[k] = sum_a wxy[a] * grid[corner_a][k] (G2 <= a few dozen values, built once per row by the warp), after which a voxel
// needs two profile reads and one lerp instead of eight grid reads.
__device__ __forceinline__ void row_profile(const double* __restrict__ grid, const size_t (&o4)[4], const double (&wxy)[4], int G2,
                                            int lane, double* __restrict__ prof) {
  for (int k = lane; k < G2; k += 32)
    prof[k] = wxy[0] * grid[o4[0] + k] + wxy[1] * grid[o4[1] + k] + wxy[2] * grid[o4[2] + k] + wxy[3] * grid[o4[3] + k];
}

// grid (X, ceil(Y / 8)), block 8 y-rows x 32 z-lanes (one warp per row, z coalesced); dynamic smem 8 x 2 x G2 doubles
__global__ void __launch_bounds__(256) s1_grid_zoom_kernel(const double* __restrict__ mean_grid, const double* __restrict__ std_grid,
                                                           GridGeom q, float* __restrict__ mean_out, float* __restrict__ std_out) {
  extern __shared__ double prof_all[];
  const int x = blockIdx.x, w = threadIdx.x >> 5, y = blockIdx.y * 8 + w, lane = threadIdx.x & 31;
  if (y >= q.Y) return;                                              // whole warp
  const int G1 = q.g[1] + 2, G2 = q.g[2] + 2;
  double* pm = prof_all + (size_t)w * 2 * G2;
  double* ps = pm + G2;
  int i0, j0; double fx, fy;
  zoom_coord(x, q.st[0], q.g[0], q.scale[0], i0, fx); zoom_coord(y, q.st[1], q.g[1], q.scale[1], j0, fy);
  const double wxy[4] = {(1 - fx) * (1 - fy), (1 - fx) * fy, fx * (1 - fy), fx * fy};
  const size_t o4[4] = {((size_t)i0 * G1 + j0) * G2, ((size_t)i0 * G1 + j0 + 1) * G2, ((size_t)(i0 + 1) * G1 + j0) * G2,
                        ((size_t)(i0 + 1) * G1 + j0 + 1) * G2};
  row_profile(mean_grid, o4, wxy, G2, lane, pm);
  if (std_out) row_profile(std_grid, o4, wxy, G2, lane, ps);
  __syncwarp();
  const int64_t row = ((int64_t)x * q.Y + y) * q.Z;
  for (int z = lane; z < q.Z; z += 32) {
    int k0; double fz;
    zoom_coord(z, q.st[2], q.g[2], q.scale[2], k0, fz);
    mean_out[row + z] = (float)(pm[k0] * (1 - fz) + pm[k0 + 1] * fz);
    if (std_out) std_out[row + z] = (float)(ps[k0] * (1 - fz) + ps[k0 + 1] * fz);
  }
}

__global__ void __launch_bounds__(256) s1_align_kernel(float* __restrict__ x, const float* __restrict__ mu_i,
                                                       const float* __restrict__ mu_p, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    x[i] = (float)(((double)x[i] - (double)mu_i[i]) + (double)mu_p[i]);
}

// lesion_analysis.py:163-169 in one launch: volume 0 is the target (its zoomed local mean is written to mu_out,
// if given), volumes >= 1 the references, aligned in place: x_i = (x_i - zoom(grid_i)) + zoom(grid_target), evaluated from
// the two coarse grids in fp64 -- the references' local-mean volumes are never materialised.
__global__ void __launch_bounds__(256) s1_zoom_align_kernel(const double* __restrict__ mean_grids, size_t grid_stride, GridGeom q,
                                                            VolPtrs vols, int nvol, float* __restrict__ mu_out) {
  // dynamic smem: per-warp profiles [8][2][G2] doubles, then the z tables fz[Z] (double) and k0[Z] (int) shared by the CTA.
  // One warp per (x, y) row; the row's coordinates, corner weights and target profile are set up once and serve the
  // target and all k references (the volume loop is inside).
  extern __shared__ double prof_all[];
  const int G1 = q.g[1] + 2, G2 = q.g[2] + 2;
  double* fz_t = prof_all + 16 * G2;
  int* k0_t = reinterpret_cast<int*>(fz_t + q.Z);
  for (int z = threadIdx.x; z < q.Z; z += 256) { int k0; double fz; zoom_coord(z, q.st[2], q.g[2], q.scale[2], k0, fz); fz_t[z] = fz; k0_t[z] = k0; }
  __syncthreads();
  const int x = blockIdx.x, w = threadIdx.x >> 5, y = blockIdx.y * 8 + w, lane = threadIdx.x & 31;
  if (y >= q.Y) return;                                              // whole warp
  double* pt = prof_all + (size_t)w * 2 * G2;
  double* pr = pt + G2;
  int i0, j0; double fx, fy;
  zoom_coord(x, q.st[0], q.g[0], q.scale[0], i0, fx); zoom_coord(y, q.st[1], q.g[1], q.scale[1], j0, fy);
  const double wxy[4] = {(1 - fx) * (1 - fy), (1 - fx) * fy, fx * (1 - fy), fx * fy};
  const size_t o4[4] = {((size_t)i0 * G1 + j0) * G2, ((size_t)i0 * G1 + j0 + 1) * G2, ((size_t)(i0 + 1) * G1 + j0) * G2,
                        ((size_t)(i0 + 1) * G1 + j0 + 1) * G2};
  row_profile(mean_grids, o4, wxy, G2, lane, pt);                    // target grid
  __syncwarp();
  const int64_t row = ((int64_t)x * q.Y + y) * q.Z;
  if (mu_out)
    for (int z = lane; z < q.Z; z += 32) { const int k0 = k0_t[z]; const double fz = fz_t[z]; mu_out[row + z] = (float)(pt[k0] * (1 - fz) + pt[k0 + 1] * fz); }
  for (int vol = 1; vol < nvol; ++vol) {
    row_profile(mean_grids + (size_t)vol * grid_stride, o4, wxy, G2, lane, pr);
    __syncwarp();
    float* xr = vols.p[vol];
    for (int zb = 0; zb < q.Z; zb += 128) {                          // four loads in flight per lane
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { const int z = zb + j * 32 + lane; v[j] = z < q.Z ? xr[row + z] : 0.f; }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int z = zb + j * 32 + lane;
        if (z >= q.Z) continue;
        const int k0 = k0_t[z];
        const double fz = fz_t[z];
        const double mt = pt[k0] * (1 - fz) + pt[k0 + 1] * fz;
        xr[row + z] = (float)(((double)v[j] - (pr[k0] * (1 - fz) + pr[k0 + 1] * fz)) + mt);
      }
    }
    __syncwarp();                                                    // pr is rewritten for the next volume
  }
}

// ---------------------------------------------------------------------------------------------------------------
// group mean / population std over the K reference volumes + NLL of the target, one pass: (K + 1) x 4 B read,
// 4 .. 12 B written per voxel.
// ---------------------------------------------------------------------------------------------------------------
struct RefPtrs { const float* p[S1_MAX_REFS]; };

// Statistics are accumulated on the deviations from the first reference (exact in fp64 for fp32 data): identical
// references give sigma == 0 exactly, as numpy's two-pass std does, and every reference value is read once.
struct NllParams { double min_std; int side; int K; };
__device__ __forceinline__ void nll_finish(double x, double r0, double sd, double sdd, const NllParams& q, float mul,
                                           float& an, float& mu_f, float& sg_f) {
  const double dm = sd / q.K, mu = r0 + dm;
  double var = sdd / q.K - dm * dm;
  var = var > 0.0 ? var : 0.0;
  double sg = sqrt(var);
  sg = q.min_std < 0.0 ? sg + 1e-6 : (sg < q.min_std ? q.min_std : sg);
  double a = (x - mu) * (x - mu) / (2.0 * sg * sg) + log(sg * 2.506);
  if (a != a) a = 0.0;                                                // np.nan_to_num(nan=0.0)
  if (q.side > 0) a = x > mu ? a : 0.0;
  else if (q.side < 0) a = x < mu ? a : 0.0;
  an = (float)(a * (double)mul); mu_f = (float)mu; sg_f = (float)sg;
}

template <bool VEC>
__global__ void __launch_bounds__(256) s1_group_nll_kernel(const float* __restrict__ xp, RefPtrs refs, NllParams q,
                                                           const float* __restrict__ mul_mask, float* __restrict__ anomaly,
                                                           float* __restrict__ mu_out, float* __restrict__ sigma_out, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n4 = VEC ? n >> 2 : 0;
  for (int64_t i = tid; i < n4; i += stride) {                        // 128-bit path: 4 voxels per thread
    const float4 r0 = dwmh::ld_stream_f4(reinterpret_cast<const float4*>(refs.p[0]) + i);
    double sd[4] = {0, 0, 0, 0}, sdd[4] = {0, 0, 0, 0};
    for (int k = 1; k < q.K; ++k) {
      const float4 r = dwmh::ld_stream_f4(reinterpret_cast<const float4*>(refs.p[k]) + i);
      const double d0 = (double)r.x - (double)r0.x, d1 = (double)r.y - (double)r0.y, d2 = (double)r.z - (double)r0.z, d3 = (double)r.w - (double)r0.w;
      sd[0] += d0; sdd[0] += d0 * d0; sd[1] += d1; sdd[1] += d1 * d1; sd[2] += d2; sdd[2] += d2 * d2; sd[3] += d3; sdd[3] += d3 * d3;
    }
    const float4 x = reinterpret_cast<const float4*>(xp)[i];
    float4 m = make_float4(1.f, 1.f, 1.f, 1.f), an, mu, sg;
    if (mul_mask) m = reinterpret_cast<const float4*>(mul_mask)[i];
    nll_finish(x.x, r0.x, sd[0], sdd[0], q, m.x, an.x, mu.x, sg.x);
    nll_finish(x.y, r0.y, sd[1], sdd[1], q, m.y, an.y, mu.y, sg.y);
    nll_finish(x.z, r0.z, sd[2], sdd[2], q, m.z, an.z, mu.z, sg.z);
    nll_finish(x.w, r0.w, sd[3], sdd[3], q, m.w, an.w, mu.w, sg.w);
    if (anomaly) reinterpret_cast<float4*>(anomaly)[i] = an;
    if (mu_out) reinterpret_cast<float4*>(mu_out)[i] = mu;
    if (sigma_out) reinterpret_cast<float4*>(sigma_out)[i] = sg;
  }
  for (int64_t i = (n4 << 2) + tid; i < n; i += stride) {             // scalar path / tail
    const double r0 = (double)__ldg(refs.p[0] + i);
    double sd = 0.0, sdd = 0.0;
    for (int k = 1; k < q.K; ++k) { const double d = (double)__ldg(refs.p[k] + i) - r0; sd += d; sdd += d * d; }
    float an, mu, sg;
    nll_finish((double)xp[i], r0, sd, sdd, q, mul_mask ? mul_mask[i] : 1.f, an, mu, sg);
    if (anomaly) anomaly[i] = an;
    if (mu_out) mu_out[i] = mu;
    if (sigma_out) sigma_out[i] = sg;
  }
}

// group_mean / group_std with per-reference masks (image_ops.py:197-231: masked values become NaN, np.nanmean / np.nanstd
// over the rest; the Otsu branch of nll, lesion_analysis.py:87-92).  A voxel no reference covers has mu = sigma = NaN and,
// after np.nan_to_num, anomaly 0.
__global__ void __launch_bounds__(256) s1_group_nll_masked_kernel(const float* __restrict__ xp, RefPtrs refs, RefPtrs masks, NllParams q,
                                                                  const float* __restrict__ mul_mask, float* __restrict__ anomaly,
                                                                  float* __restrict__ mu_out, float* __restrict__ sigma_out, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    double r0 = 0.0, sd = 0.0, sdd = 0.0;
    int cnt = 0;
    for (int k = 0; k < q.K; ++k) {
      if (__ldg(masks.p[k] + i) < 0.5f) continue;                    // np.where(mask < 0.5, nan, data)
      const double r = (double)__ldg(refs.p[k] + i);
      if (cnt == 0) r0 = r;
      else { const double d = r - r0; sd += d; sdd += d * d; }
      ++cnt;
    }
    float an, mu, sg;
    if (cnt == 0) {
      an = 0.f * (mul_mask ? mul_mask[i] : 1.f);
      mu = sg = __int_as_float(0x7fc00000);
    } else {
      NllParams qq = q; qq.K = cnt;
      nll_finish((double)xp[i], r0, sd, sdd, qq, mul_mask ? mul_mask[i] : 1.f, an, mu, sg);
    }
    if (anomaly) anomaly[i] = an;
    if (mu_out) mu_out[i] = mu;
    if (sigma_out) sigma_out[i] = sg;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// median filter, scipy.ndimage.median_filter(size=(kx,ky,kz), mode='constant', cval=0): window [i - k/2, i - k/2 + k)
// per axis, rank (kx ky kz) / 2 of the ascending window.  One thread per voxel, CTA tile 2 x 4 x 32 (z fastest) staged
// with its halo in shared memory as order-preserving integer keys; the rank is found by a 32-step bitwise search on
// the key (count of window keys below the probe), so any window size costs 32 N shared-memory reads and no sort.
// ---------------------------------------------------------------------------------------------------------------
constexpr int MT_X = 2, MT_Y = 4, MT_Z = 32;

__device__ __forceinline__ uint32_t f2key(float f) { const uint32_t u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float key2f(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

__global__ void __launch_bounds__(256) s1_median_kernel(const float* __restrict__ in, float* __restrict__ out, int X, int Y, int Z,
                                                        int kx, int ky, int kz) {
  extern __shared__ uint32_t tile[];
  const int tx = MT_X + kx - 1, ty = MT_Y + ky - 1, tz = MT_Z + kz - 1;
  const int bz = blockIdx.x * MT_Z, by = blockIdx.y * MT_Y, bx = blockIdx.z * MT_X;
  const int ox = bx - kx / 2, oy = by - ky / 2, oz = bz - kz / 2;
  for (int t = threadIdx.x; t < tx * ty * tz; t += blockDim.x) {
    const int c = t % tz, b = (t / tz) % ty, a = t / (tz * ty);
    const int gx = ox + a, gy = oy + b, gz = oz + c;
    float v = 0.f;                                                   // cval
    if (gx >= 0 && gx < X && gy >= 0 && gy < Y && gz >= 0 && gz < Z) v = in[((int64_t)gx * Y + gy) * Z + gz];
    tile[t] = f2key(v);
  }
  __syncthreads();
  const int lz = threadIdx.x % MT_Z, ly = (threadIdx.x / MT_Z) % MT_Y, lx = threadIdx.x / (MT_Z * MT_Y);
  const int gx = bx + lx, gy = by + ly, gz = bz + lz;
  if (gx >= X || gy >= Y || gz >= Z) return;
  const int rank = (kx * ky * kz) / 2;
  uint32_t key = 0;
  for (int bit = 31; bit >= 0; --bit) {
    const uint32_t probe = key | (1u << bit);
    int below = 0;
    for (int a = 0; a < kx; ++a)
      for (int b = 0; b < ky; ++b) {
        const uint32_t* row = tile + ((lx + a) * ty + (ly + b)) * tz + lz;
        for (int c = 0; c < kz; ++c) below += row[c] < probe ? 1 : 0;
      }
    if (below <= rank) key = probe;                                  // largest key with (#window keys below it) <= rank
  }
  out[((int64_t)gx * Y + gy) * Z + gz] = key2f(key);
}

// Compile-time windows up to 65 values (3x3x3 = the 1 mm isotropic case; k x k slices for thick-slice data): the
// window goes through registers once and the median is found by forgetful selection -- of N/2 + 2 values neither the
// minimum nor the maximum can be the median, so drop both, add the next value, repeat -- with min/max exchanges only
// (~155 exchanges for N = 27 instead of 32 x 27 compares).
template <int S, int W>
__device__ __forceinline__ void minmax_ends(uint32_t (&v)[W]) {     // min of v[0..S) -> v[0], max -> v[S-1]
#pragma unroll
  for (int i = 0; i < S / 2; ++i) { const uint32_t lo = min(v[i], v[S - 1 - i]), hi = max(v[i], v[S - 1 - i]); v[i] = lo; v[S - 1 - i] = hi; }
#pragma unroll
  for (int i = 1; i <= (S - 1) / 2; ++i) { const uint32_t lo = min(v[0], v[i]), hi = max(v[0], v[i]); v[0] = lo; v[i] = hi; }
#pragma unroll
  for (int i = S / 2; i < S - 1; ++i) { const uint32_t lo = min(v[i], v[S - 1]), hi = max(v[i], v[S - 1]); v[i] = lo; v[S - 1] = hi; }
}
template <int KY, int KZ, int N>
__device__ __forceinline__ uint32_t window_key(const uint32_t* __restrict__ base, int ty, int tz, int e) {
  return e < N ? base[((e / (KY * KZ)) * ty + (e / KZ) % KY) * tz + e % KZ] : 0xffffffffu;   // e >= N: the +inf pad of even windows
}
template <int S, int W, int NP, int N, int KY, int KZ>
__device__ __forceinline__ void forget_step(uint32_t (&v)[W], const uint32_t* __restrict__ base, int ty, int tz) {
  if constexpr (S >= 3) {
    constexpr int e = NP - (S - 2);                                  // index of the window value added at this size
    if constexpr (S < W) v[0] = window_key<KY, KZ, N>(base, ty, tz, e);
    minmax_ends<S, W>(v);
    forget_step<S - 1, W, NP, N, KY, KZ>(v, base, ty, tz);
  }
}

// Even windows (4x4x4, 6x6 slices ...): scipy takes rank N / 2 (the upper median); padding the window with one +inf key
// makes it odd without moving that rank, so the same selection applies.
template <int KX, int KY, int KZ>
__global__ void __launch_bounds__(256) s1_median_small_kernel(const float* __restrict__ in, float* __restrict__ out, int X, int Y, int Z) {
  constexpr int N = KX * KY * KZ, NP = N | 1, W = NP / 2 + 2;
  static_assert(N >= 3 && N <= 65, "windows of 3..65 values");
  constexpr int tx = MT_X + KX - 1, ty = MT_Y + KY - 1, tz = MT_Z + KZ - 1;
  __shared__ uint32_t tile[tx * ty * tz];
  const int bz = blockIdx.x * MT_Z, by = blockIdx.y * MT_Y, bx = blockIdx.z * MT_X;
  const int ox = bx - KX / 2, oy = by - KY / 2, oz = bz - KZ / 2;
  for (int t = threadIdx.x; t < tx * ty * tz; t += 256) {
    const int c = t % tz, b = (t / tz) % ty, a = t / (tz * ty);
    const int gx = ox + a, gy = oy + b, gz = oz + c;
    float v = 0.f;
    if (gx >= 0 && gx < X && gy >= 0 && gy < Y && gz >= 0 && gz < Z) v = in[((int64_t)gx * Y + gy) * Z + gz];
    tile[t] = f2key(v);
  }
  __syncthreads();
  const int lz = threadIdx.x % MT_Z, ly = (threadIdx.x / MT_Z) % MT_Y, lx = threadIdx.x / (MT_Z * MT_Y);
  const int gx = bx + lx, gy = by + ly, gz = bz + lz;
  if (gx >= X || gy >= Y || gz >= Z) return;
  const uint32_t* base = tile + (lx * ty + ly) * tz + lz;
  uint32_t v[W];
#pragma unroll
  for (int e = 0; e < W; ++e) v[e] = window_key<KY, KZ, N>(base, ty, tz, e);
  forget_step<W, W, NP, N, KY, KZ>(v, base, ty, tz);                 // ends with the median of the last three in v[1]
  out[((int64_t)gx * Y + gy) * Z + gz] = key2f(v[1]);
}

template <int KX, int KY, int KZ>
bool median_small_launch(int kx, int ky, int kz, dim3 grid, cudaStream_t st, const float* in, float* out, int X, int Y, int Z) {
  if (kx != KX || ky != KY || kz != KZ) return false;
  s1_median_small_kernel<KX, KY, KZ><<<grid, 256, 0, st>>>(in, out, X, Y, Z);
  return true;
}

// ---------------------------------------------------------------------------------------------------------------
// component_filtering (image_ops.py:253-306).  Per filtered orientation `ax`: 2-D binary erosion of every slice
// (scipy's cross, border = background) fused into the label initialisation, union-find over the two in-plane axes
// (roots = smallest voxel index = scipy's raster label order), component sizes, per-slice winner by a packed 64-bit
// atomicMax {size, ~root} (largest component, first label on ties), membership added to the running sum `acc`.
// Orientations that are not filtered add the mask itself; the result is acc > 0.5.
// ---------------------------------------------------------------------------------------------------------------
struct Dims { int n[3]; int64_t stride[3]; };
__device__ __forceinline__ void cf_coords(int64_t v, const Dims& d, int (&c)[3]) {
  c[2] = (int)(v % d.n[2]); c[1] = (int)((v / d.n[2]) % d.n[1]); c[0] = (int)(v / ((int64_t)d.n[2] * d.n[1]));
}

__global__ void __launch_bounds__(256) cf_erode_init_kernel(const float* __restrict__ mask, int* __restrict__ L, int* __restrict__ size,
                                                            Dims d, int ax, int64_t V) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); v0 < V; v0 += stride) {   // warp-uniform trip count
    const int64_t v = v0 + (threadIdx.x & 31);
    const bool in = v < V;
    int c[3] = {0, 0, 0};
    bool keep = false;
    if (in) {
      cf_coords(v, d, c);
      keep = mask[v] != 0.f;
#pragma unroll
      for (int a = 0; a < 3; ++a)
        if (a != ax && keep)
          keep = c[a] > 0 && c[a] + 1 < d.n[a] && mask[v - d.stride[a]] != 0.f && mask[v + d.stride[a]] != 0.f;
    }
    // z-runs are components of the slice unless z is the slicing axis (then voxels along z belong to different slices)
    const int l = ax != 2 ? dwmh::ccl_run_start(keep, in && c[2] == 0, v) : (keep ? (int)v : -1);
    if (in) { L[v] = l; size[v] = 0; }
  }
}

__global__ void __launch_bounds__(256) cf_merge_kernel(int* __restrict__ L, Dims d, int ax, int64_t V) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) {
    if (L[v] < 0) continue;
    int c[3];
    cf_coords(v, d, c);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (a == ax || c[a] + 1 >= d.n[a] || L[v + d.stride[a]] < 0) continue;
      if (a == 2 && ((v + 1) & 31) != 0) continue;                   // linked by the run initialisation
      dwmh::ccl_union(L, (int)v, (int)(v + d.stride[a]));
    }
  }
}

__global__ void __launch_bounds__(256) cf_best_kernel(const int* __restrict__ L, const int* __restrict__ size,
                                                      unsigned long long* __restrict__ best, Dims d, int ax, int64_t V) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) {
    if (L[v] != (int)v) continue;                                    // component roots only
    int c[3];
    cf_coords(v, d, c);
    atomicMax(best + c[ax], ((unsigned long long)(unsigned)size[v] << 32) | (unsigned long long)(0xffffffffu - (unsigned)v));
  }
}

__global__ void __launch_bounds__(256) cf_accum_kernel(const int* __restrict__ L, const unsigned long long* __restrict__ best,
                                                       float* __restrict__ acc, Dims d, int ax, int64_t V) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) {
    const int r = L[v];
    if (r < 0) continue;
    int c[3];
    cf_coords(v, d, c);
    const unsigned long long b = best[c[ax]];
    if (b != 0ull && (unsigned)r == 0xffffffffu - (unsigned)(b & 0xffffffffull)) acc[v] += 1.f;
  }
}

__global__ void __launch_bounds__(256) cf_passthrough_kernel(const float* __restrict__ mask, float* __restrict__ acc, int64_t V) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) acc[v] += mask[v];
}

__global__ void __launch_bounds__(256) cf_final_kernel(const float* __restrict__ acc, float* __restrict__ out, int64_t V) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) out[v] = acc[v] > 0.5f ? 1.f : 0.f;
}

// ---------------------------------------------------------------------------------------------------------------
// Otsu threshold support (skimage.filters.threshold_otsu as called at lesion_analysis.py:145-146 and image_ops.py:308-323):
// min / max over a mask, and numpy.histogram's equal-width binning with its exact edge corrections (bin i holds
// edges[i] <= v < edges[i+1], the last bin is closed); the 256-entry Otsu scan itself runs on the host.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) s1_minmax_kernel(const float* __restrict__ x, const float* __restrict__ mask, int64_t n,
                                                        int* __restrict__ mm) {       // mm[0] = min, mm[1] = max (ordered ints)
  int mn = 0x7fffffff, mx = (int)0x80000000;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    if (!mask || mask[i] > 0.5f) { const int o = f2ord(x[i]); mn = min(mn, o); mx = max(mx, o); }
  mn = __reduce_min_sync(0xffffffffu, mn); mx = __reduce_max_sync(0xffffffffu, mx);
  if ((threadIdx.x & 31) == 0) { atomicMin(mm, mn); atomicMax(mm + 1, mx); }
}

// voxels outside the mask count as `fill` (np.where(mask < 0.5, fill, x)) when fill_outside, else they are skipped
__global__ void __launch_bounds__(256) s1_histogram_kernel(const float* __restrict__ x, const float* __restrict__ mask, int64_t n,
                                                           int fill_outside, float fill, const double* __restrict__ edges, int nbins,
                                                           unsigned long long* __restrict__ counts) {
  extern __shared__ unsigned char hsm[];
  double* e = reinterpret_cast<double*>(hsm);                         // [nbins + 1]
  unsigned int* h = reinterpret_cast<unsigned int*>(e + nbins + 1);   // [nbins]
  for (int i = threadIdx.x; i <= nbins; i += blockDim.x) e[i] = edges[i];
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) h[i] = 0u;
  __syncthreads();
  const double first = e[0], last = e[nbins], norm = (double)nbins / (last - first);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float v = x[i];
    if (mask) {                                                       // data[mask > 0.5]  vs  np.where(mask < 0.5, fill, data)
      const float m = mask[i];
      if (fill_outside) { if (m < 0.5f) v = fill; }
      else if (!(m > 0.5f)) continue;
    }
    const double d = (double)v;
    if (!(d >= first && d <= last)) continue;                         // outside the range (and NaN): not counted
    int b = (int)((d - first) * norm);
    b = b < 0 ? 0 : (b > nbins - 1 ? nbins - 1 : b);
    if (d < e[b]) --b;
    else if (b != nbins - 1 && d >= e[b + 1]) ++b;
    atomicAdd(&h[b], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) if (h[i]) atomicAdd(counts + i, (unsigned long long)h[i]);
}

__global__ void __launch_bounds__(256) s1_threshold_kernel(const float* __restrict__ x, float thr, const float* __restrict__ mul,
                                                           float* __restrict__ out, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = (x[i] > thr ? 1.f : 0.f) * (mul ? mul[i] : 1.f);
}

// ---------------------------------------------------------------------------------------------------------------
// Tissue priors of nll_analysis (lesion_analysis.py:213-243): majority vote over the K registered label maps
// (average_contiguous_labels, image_ops.py:23-38: per-voxel argmax of the label histogram, first maximum wins), the
// "labelled as tissue by more than half of the references" mask, and their application to the anomaly score.
// ---------------------------------------------------------------------------------------------------------------
constexpr int S1_MAX_LABELS = 16;
__global__ void __launch_bounds__(256) s1_label_vote_kernel(RefPtrs labels, int K, int nch, float* __restrict__ avg_label,
                                                            float* __restrict__ tissue_majority, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    unsigned long long votes = 0ull, votes_hi = 0ull;                // 2 x 8 label ids, one 8-bit counter each (K <= 32)
    int tissue = 0;
    for (int k = 0; k < K; ++k) {
      const float t = __ldg(labels.p[k] + i);
      const int c = (int)t;                                          // label.astype('int')
      if (c >= 0 && c < 8) votes += 1ull << (8 * c);
      else if (c >= 8 && c < nch) votes_hi += 1ull << (8 * (c - 8));
      tissue += t > 0.5f ? 1 : 0;
    }
    int best = 0, best_n = -1;
    for (int c = 0; c < nch; ++c) {
      const int v = (int)(((c < 8 ? votes >> (8 * c) : votes_hi >> (8 * (c - 8)))) & 0xffull);
      if (v > best_n) { best_n = v; best = c; }
    }
    if (avg_label) avg_label[i] = (float)best;
    if (tissue_majority) tissue_majority[i] = (2 * tissue > K) ? 1.f : 0.f;   // tissue_sum > sample_size / 2
  }
}

// stage 1: a *= (avg_label > 0.5)                                           (:216)
// stage 2: a = (1.5 < avg_label < 2.5 ? a_median : a) * tissue_majority      (:232-243)
__global__ void __launch_bounds__(256) s1_apply_priors_kernel(float* __restrict__ a, const float* __restrict__ a_median,
                                                              const float* __restrict__ avg_label, const float* __restrict__ tissue_majority,
                                                              int stage, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float l = avg_label[i];
    if (stage == 1) a[i] = l > 0.5f ? a[i] : 0.f * a[i];
    else a[i] = ((l > 1.5f && l < 2.5f) ? a_median[i] : a[i]) * tissue_majority[i];
  }
}

int geom(int X, int Y, int Z, const int32_t patch[3], GridGeom* q) {
  if (X <= 0 || Y <= 0 || Z <= 0) return fail("mean_std_grid: empty volume");
  q->X = X; q->Y = Y; q->Z = Z;
  const int sh[3] = {X, Y, Z};
  for (int a = 0; a < 3; ++a) {
    if (patch[a] <= 0) return fail("mean_std_grid: patch_size[%d] = %d", a, patch[a]);
    const int ps = 2 * ((patch[a] + 1) / 2);                         // 2 * ceil(p / 2)
    q->st[a] = ps / 2;
    q->pad[a] = ps * ((sh[a] + ps - 1) / ps);
    q->g[a] = q->pad[a] / q->st[a];
    q->scale[a] = (double)(q->g[a] + 1) / (double)((q->g[a] + 2) * q->st[a] - 1);
  }
  return 0;
}
size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
int cs_threads(int Z) { const int t = (Z + 31) & ~31; return t < 256 ? t : 256; }   // one thread per z, whole warps

}  // namespace

static int zscore_launch(int device, VolPtrs vols, int nvol, const float* mask, int64_t n, int fill_outside, void* workspace,
                         bool aligned, cudaStream_t st) {
  double* ws = (double*)workspace;
  CU_TRY(cudaMemsetAsync(ws, 0, (size_t)nvol * ZS_SLOT * sizeof(double), st));
  // min slot <- 0x7f7f7f7f (above the key of every float below 3.39e38): one strided 2-D memset over the slots
  CU_TRY(cudaMemset2DAsync((char*)workspace + 32, ZS_SLOT * sizeof(double), 0x7f, 4, nvol, st));
  const dim3 grid((sm_count(device) * 8 + nvol - 1) / nvol, nvol);
  if (aligned) {
    s1_stats_kernel<true><<<grid, 256, 0, st>>>(vols, mask, n, ws);
    s1_zscore_apply_kernel<true><<<grid, 256, 0, st>>>(vols, mask, n, ws, fill_outside);
  } else {
    s1_stats_kernel<false><<<grid, 256, 0, st>>>(vols, mask, n, ws);
    s1_zscore_apply_kernel<false><<<grid, 256, 0, st>>>(vols, mask, n, ws, fill_outside);
  }
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_zscore(int32_t device, float* x, const float* mask, int64_t n, int32_t fill_outside, void* workspace,
                              double* stats_out, void* stream_) {
  if (!x || !workspace) return fail("dwmh_s1_zscore: null argument");
  if (n <= 0) return fail("dwmh_s1_zscore: empty volume");
  if (fill_outside && !mask) return fail("dwmh_s1_zscore: fill_outside needs a mask");
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(device);
  VolPtrs vols{}; vols.p[0] = x;
  if (zscore_launch(device, vols, 1, mask, n, fill_outside, workspace, (((uintptr_t)x | (uintptr_t)mask) & 15) == 0, st)) return 1;
  if (stats_out) {
    double h[4];
    CU_TRY(cudaMemcpyAsync(h, workspace, sizeof h, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    const double cnt = h[2] > 0 ? h[2] : 1.0, m = h[0] / cnt;
    double var = h[1] / cnt - m * m; if (var < 0) var = 0;
    stats_out[0] = m; stats_out[1] = sqrt(var); stats_out[2] = h[2];
  }
  return 0;
}

extern "C" int dwmh_s1_zscore_batch(int32_t device, float* const* xs, int32_t nvol, const float* mask, int64_t n, int32_t fill_outside,
                                    void* workspace, void* stream_) {
  if (!xs || !workspace) return fail("dwmh_s1_zscore_batch: null argument");
  if (nvol <= 0 || nvol > S1_MAX_VOLS) return fail("dwmh_s1_zscore_batch: %d volumes (1..%d supported)", nvol, S1_MAX_VOLS);
  if (n <= 0) return fail("dwmh_s1_zscore_batch: empty volume");
  if (fill_outside && !mask) return fail("dwmh_s1_zscore_batch: fill_outside needs a mask");
  VolPtrs vols{};
  uintptr_t al = (uintptr_t)mask;
  for (int i = 0; i < nvol; ++i) { if (!xs[i]) return fail("dwmh_s1_zscore_batch: xs[%d] is null", i); vols.p[i] = xs[i]; al |= (uintptr_t)xs[i]; }
  DEV_GUARD(device);
  return zscore_launch(device, vols, nvol, mask, n, fill_outside, workspace, (al & 15) == 0, (cudaStream_t)stream_);
}

extern "C" int dwmh_s1_mean_std_grid_workspace(int32_t X, int32_t Y, int32_t Z, const int32_t patch_size[3], int64_t* bytes) {
  GridGeom q;
  if (!patch_size || !bytes) return fail("dwmh_s1_mean_std_grid_workspace: null argument");
  if (geom(X, Y, Z, patch_size, &q)) return 1;
  const size_t cells = (size_t)q.g[0] * q.g[1] * q.g[2], grid = (size_t)(q.g[0] + 2) * (q.g[1] + 2) * (q.g[2] + 2);
  *bytes = (int64_t)(align256(cells * 3 * sizeof(double)) + 2 * align256(grid * sizeof(double)));
  return 0;
}

extern "C" int dwmh_s1_mean_std_grid(int32_t device, const float* x, const float* mask, int32_t X, int32_t Y, int32_t Z,
                                     const int32_t patch_size[3], float* mean_out, float* std_out, void* workspace, void* stream_) {
  if (!x || !mean_out || !workspace || !patch_size) return fail("dwmh_s1_mean_std_grid: null argument");
  GridGeom q;
  if (geom(X, Y, Z, patch_size, &q)) return 1;
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(device);
  const size_t ncell = (size_t)q.g[0] * q.g[1] * q.g[2], ngrid = (size_t)(q.g[0] + 2) * (q.g[1] + 2) * (q.g[2] + 2);
  double* cells = (double*)workspace;
  double* mg = (double*)((char*)workspace + align256(ncell * 3 * sizeof(double)));
  double* sg = (double*)((char*)mg + align256(ngrid * sizeof(double)));
  CU_TRY(cudaMemsetAsync(workspace, 0, align256(ncell * 3 * sizeof(double)) + 2 * align256(ngrid * sizeof(double)), st));
  const int slabs = (q.st[0] + CS_SLAB - 1) / CS_SLAB;
  if (q.g[2] > 300) return fail("dwmh_s1_mean_std_grid: %d cells along z exceed the shared-memory tables (300)", q.g[2]);
  VolPtrs vols{}; vols.p[0] = const_cast<float*>(x);
  s1_cell_sums_kernel<<<(unsigned)(q.g[0] * q.g[1] * slabs), cs_threads(Z), 3 * cs_threads(Z) * sizeof(double), st>>>(vols, mask, q, slabs, cells);
  s1_grid_stats_kernel<<<(unsigned)((ncell + 127) / 128), 128, 0, st>>>(cells, q, mask ? 1 : 0, mg, sg, 0);
  if ((Y + 7) / 8 > 65535) return fail("dwmh_s1_mean_std_grid: volume too large");
  s1_grid_zoom_kernel<<<dim3(X, (Y + 7) / 8), 256, 16 * (q.g[2] + 2) * sizeof(double), st>>>(mg, sg, q, mean_out, std_out);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_local_mean_align_workspace(int32_t X, int32_t Y, int32_t Z, const int32_t patch_size[3], int32_t k, int64_t* bytes) {
  GridGeom q;
  if (!patch_size || !bytes) return fail("dwmh_s1_local_mean_align_workspace: null argument");
  if (k < 0 || k > S1_MAX_REFS) return fail("dwmh_s1_local_mean_align_workspace: k = %d (0..%d supported)", k, S1_MAX_REFS);
  if (geom(X, Y, Z, patch_size, &q)) return 1;
  const size_t cells = (size_t)q.g[0] * q.g[1] * q.g[2], grid = (size_t)(q.g[0] + 2) * (q.g[1] + 2) * (q.g[2] + 2);
  *bytes = (int64_t)(align256((size_t)(k + 1) * cells * 3 * sizeof(double)) + 2 * (size_t)(k + 1) * align256(grid * sizeof(double)));
  return 0;
}

extern "C" int dwmh_s1_local_mean_align(int32_t device, const float* target, float* const* refs, int32_t k, const float* mask,
                                        int32_t X, int32_t Y, int32_t Z, const int32_t patch_size[3], float* target_local_mu_out,
                                        void* workspace, void* stream_) {
  if (!target || !workspace || !patch_size || (k > 0 && !refs)) return fail("dwmh_s1_local_mean_align: null argument");
  if (k < 0 || k > S1_MAX_REFS) return fail("dwmh_s1_local_mean_align: k = %d reference images (0..%d supported)", k, S1_MAX_REFS);
  GridGeom q;
  if (geom(X, Y, Z, patch_size, &q)) return 1;
  if (q.g[2] > 300) return fail("dwmh_s1_local_mean_align: %d cells along z exceed the shared-memory tables (300)", q.g[2]);
  if ((Y + 7) / 8 > 65535) return fail("dwmh_s1_local_mean_align: volume too large");
  VolPtrs vols{}; vols.p[0] = const_cast<float*>(target);
  for (int i = 0; i < k; ++i) { if (!refs[i]) return fail("dwmh_s1_local_mean_align: refs[%d] is null", i); vols.p[i + 1] = refs[i]; }
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(device);
  const int nvol = k + 1;
  const size_t ncell = (size_t)q.g[0] * q.g[1] * q.g[2], gstride = align256((size_t)(q.g[0] + 2) * (q.g[1] + 2) * (q.g[2] + 2) * sizeof(double)) / sizeof(double);
  const size_t cells_bytes = align256((size_t)nvol * ncell * 3 * sizeof(double));
  double* cells = (double*)workspace;
  double* mg = (double*)((char*)workspace + cells_bytes);
  double* sg = mg + (size_t)nvol * gstride;
  CU_TRY(cudaMemsetAsync(workspace, 0, cells_bytes + 2 * (size_t)nvol * gstride * sizeof(double), st));
  const int slabs = (q.st[0] + CS_SLAB - 1) / CS_SLAB;
  s1_cell_sums_kernel<<<dim3((unsigned)(q.g[0] * q.g[1] * slabs), nvol), cs_threads(Z), 3 * cs_threads(Z) * sizeof(double), st>>>(vols, mask, q, slabs, cells);
  s1_grid_stats_kernel<<<dim3((unsigned)((ncell + 127) / 128), nvol), 128, 0, st>>>(cells, q, mask ? 1 : 0, mg, sg, gstride);
  const size_t za_smem = 16 * (size_t)(q.g[2] + 2) * sizeof(double) + (size_t)Z * (sizeof(double) + sizeof(int));
  if (za_smem > 48 * 1024) return fail("dwmh_s1_local_mean_align: Z = %d exceeds the shared-memory z table", Z);
  s1_zoom_align_kernel<<<dim3(X, (Y + 7) / 8), 256, za_smem, st>>>(mg, gstride, q, vols, nvol, target_local_mu_out);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_align_local_mean(int32_t device, float* x, const float* local_mu, const float* target_local_mu, int64_t n, void* stream_) {
  if (!x || !local_mu || !target_local_mu) return fail("dwmh_s1_align_local_mean: null argument");
  DEV_GUARD(device);
  s1_align_kernel<<<sm_count(device) * 8, 256, 0, (cudaStream_t)stream_>>>(x, local_mu, target_local_mu, n);
  CU_TRY(cudaGetLastError());
  return 0;
}

static int group_nll_impl(const char* who, int32_t device, const float* x_prime, const float* const* refs, const float* const* masks, int32_t k,
                          double min_std, int32_t side, const float* mul_mask, float* anomaly, float* mu_out, float* sigma_out, int64_t n,
                          void* stream_) {
  if (!x_prime || !refs) return fail("%s: null argument", who);
  if (k <= 0 || k > S1_MAX_REFS) return fail("%s: k = %d reference images (1..%d supported)", who, k, S1_MAX_REFS);
  if (side < -1 || side > 1) return fail("%s: side must be -1, 0 or +1", who);
  RefPtrs rp{}, mp{};
  for (int i = 0; i < k; ++i) {
    if (!refs[i] || (masks && !masks[i])) return fail("%s: refs[%d] / masks[%d] is null", who, i, i);
    rp.p[i] = refs[i];
    if (masks) mp.p[i] = masks[i];
  }
  DEV_GUARD(device);
  const NllParams q{min_std, side, k};
  cudaStream_t st = (cudaStream_t)stream_;
  if (masks) {
    s1_group_nll_masked_kernel<<<sm_count(device) * 8, 256, 0, st>>>(x_prime, rp, mp, q, mul_mask, anomaly, mu_out, sigma_out, n);
  } else {
    uintptr_t al = (uintptr_t)x_prime | (uintptr_t)mul_mask | (uintptr_t)anomaly | (uintptr_t)mu_out | (uintptr_t)sigma_out;
    for (int i = 0; i < k; ++i) al |= (uintptr_t)refs[i];
    if ((al & 15) == 0) s1_group_nll_kernel<true><<<sm_count(device) * 8, 256, 0, st>>>(x_prime, rp, q, mul_mask, anomaly, mu_out, sigma_out, n);
    else s1_group_nll_kernel<false><<<sm_count(device) * 8, 256, 0, st>>>(x_prime, rp, q, mul_mask, anomaly, mu_out, sigma_out, n);
  }
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_group_nll(int32_t device, const float* x_prime, const float* const* refs, int32_t k, double min_std, int32_t side,
                                 const float* mul_mask, float* anomaly, float* mu_out, float* sigma_out, int64_t n, void* stream_) {
  return group_nll_impl("dwmh_s1_group_nll", device, x_prime, refs, nullptr, k, min_std, side, mul_mask, anomaly, mu_out, sigma_out, n, stream_);
}

extern "C" int dwmh_s1_group_nll_masked(int32_t device, const float* x_prime, const float* const* refs, const float* const* ref_masks, int32_t k,
                                        double min_std, int32_t side, const float* mul_mask, float* anomaly, float* mu_out, float* sigma_out,
                                        int64_t n, void* stream_) {
  if (!ref_masks) return fail("dwmh_s1_group_nll_masked: null argument");
  return group_nll_impl("dwmh_s1_group_nll_masked", device, x_prime, refs, ref_masks, k, min_std, side, mul_mask, anomaly, mu_out, sigma_out, n, stream_);
}

extern "C" int dwmh_s1_median_filter(int32_t device, const float* in, float* out, int32_t X, int32_t Y, int32_t Z,
                                     const int32_t kernel_size[3], void* stream_) {
  if (!in || !out || !kernel_size) return fail("dwmh_s1_median_filter: null argument");
  if (in == out) return fail("dwmh_s1_median_filter: in and out must not alias");
  if (X <= 0 || Y <= 0 || Z <= 0) return fail("dwmh_s1_median_filter: empty volume");
  const int kx = kernel_size[0], ky = kernel_size[1], kz = kernel_size[2];
  if (kx < 1 || ky < 1 || kz < 1 || kx > 9 || ky > 9 || kz > 9) return fail("dwmh_s1_median_filter: kernel %dx%dx%d (1..9 per axis supported)", kx, ky, kz);
  DEV_GUARD(device);
  const size_t smem = (size_t)(MT_X + kx - 1) * (MT_Y + ky - 1) * (MT_Z + kz - 1) * sizeof(uint32_t);
  dim3 grid((Z + MT_Z - 1) / MT_Z, (Y + MT_Y - 1) / MT_Y, (X + MT_X - 1) / MT_X);
  if (grid.y > 65535 || grid.z > 65535) return fail("dwmh_s1_median_filter: volume too large");
  cudaStream_t st = (cudaStream_t)stream_;
  // register-resident selection for the windows median_3mm produces at common resolutions: 1 mm isotropic (3x3x3),
  // ~0.75 mm (4x4x4), thick slices with 1 / 0.75 / 0.6 / 0.5 mm in-plane (3x3, 4x4, 5x5, 6x6 across any axis)
#define MS(a, b, c) median_small_launch<a, b, c>(kx, ky, kz, grid, st, in, out, X, Y, Z)
  const bool done = MS(3, 3, 3) || MS(4, 4, 4) || MS(1, 3, 3) || MS(3, 1, 3) || MS(3, 3, 1) || MS(1, 4, 4) || MS(4, 1, 4) || MS(4, 4, 1) ||
                    MS(1, 5, 5) || MS(5, 1, 5) || MS(5, 5, 1) || MS(1, 6, 6) || MS(6, 1, 6) || MS(6, 6, 1);
#undef MS
  if (!done) s1_median_kernel<<<grid, 256, smem, st>>>(in, out, X, Y, Z, kx, ky, kz);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_component_filtering_workspace(int32_t X, int32_t Y, int32_t Z, int64_t* bytes) {
  if (!bytes) return fail("dwmh_s1_component_filtering_workspace: null argument");
  if (X <= 0 || Y <= 0 || Z <= 0) return fail("dwmh_s1_component_filtering_workspace: empty volume");
  const size_t V = (size_t)X * Y * Z, m = (size_t)(X > Y ? (X > Z ? X : Z) : (Y > Z ? Y : Z));
  *bytes = (int64_t)(3 * align256(V * 4) + align256(m * 8));
  return 0;
}

extern "C" int dwmh_s1_component_filtering(int32_t device, const float* mask, int32_t X, int32_t Y, int32_t Z, const double voxel_size[3],
                                           float* out, void* workspace, void* stream_) {
  if (!mask || !out || !workspace || !voxel_size) return fail("dwmh_s1_component_filtering: null argument");
  if (X <= 0 || Y <= 0 || Z <= 0) return fail("dwmh_s1_component_filtering: empty volume");
  const int64_t V = (int64_t)X * Y * Z;
  if (V >= (int64_t)1 << 31) return fail("dwmh_s1_component_filtering: volume of %lld voxels exceeds the 32-bit label range", (long long)V);
  for (int a = 0; a < 3; ++a) if (!(voxel_size[a] > 0.0)) return fail("dwmh_s1_component_filtering: voxel_size[%d] must be positive", a);
  // thick-slice data (max / min > 3): only the slices across the thick axis are filtered (np.argmax: first maximum)
  const double mx = fmax(voxel_size[0], fmax(voxel_size[1], voxel_size[2])), mn = fmin(voxel_size[0], fmin(voxel_size[1], voxel_size[2]));
  bool filt[3] = {true, true, true};
  if (mx / mn > 3.0) {
    const int am = voxel_size[0] >= voxel_size[1] ? (voxel_size[0] >= voxel_size[2] ? 0 : 2) : (voxel_size[1] >= voxel_size[2] ? 1 : 2);
    for (int a = 0; a < 3; ++a) filt[a] = a == am;
  }
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(device);
  int* L = (int*)workspace;
  int* size = (int*)((char*)workspace + align256((size_t)V * 4));
  float* acc = (float*)((char*)workspace + 2 * align256((size_t)V * 4));
  unsigned long long* best = (unsigned long long*)((char*)workspace + 3 * align256((size_t)V * 4));
  const Dims d{{X, Y, Z}, {(int64_t)Y * Z, (int64_t)Z, 1}};
  const int grid = sm_count(device) * 8;
  CU_TRY(cudaMemsetAsync(acc, 0, (size_t)V * 4, st));
  for (int ax = 0; ax < 3; ++ax) {
    if (!filt[ax]) { cf_passthrough_kernel<<<grid, 256, 0, st>>>(mask, acc, V); continue; }
    CU_TRY(cudaMemsetAsync(best, 0, (size_t)d.n[ax] * 8, st));
    cf_erode_init_kernel<<<grid, 256, 0, st>>>(mask, L, size, d, ax, V);
    cf_merge_kernel<<<grid, 256, 0, st>>>(L, d, ax, V);
    dwmh::ccl_count_kernel<<<grid, 256, 0, st>>>(L, size, V);
    cf_best_kernel<<<grid, 256, 0, st>>>(L, size, best, d, ax, V);
    cf_accum_kernel<<<grid, 256, 0, st>>>(L, best, acc, d, ax, V);
  }
  cf_final_kernel<<<grid, 256, 0, st>>>(acc, out, V);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_minmax(int32_t device, const float* x, const float* mask, int64_t n, void* workspace, float out_minmax[2], void* stream_) {
  if (!x || !workspace || !out_minmax) return fail("dwmh_s1_minmax: null argument");
  if (n <= 0) return fail("dwmh_s1_minmax: empty volume");
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(device);
  const int init[2] = {0x7fffffff, (int)0x80000000};
  int* mm = (int*)workspace;
  CU_TRY(cudaMemcpyAsync(mm, init, sizeof init, cudaMemcpyHostToDevice, st));
  s1_minmax_kernel<<<sm_count(device) * 8, 256, 0, st>>>(x, mask, n, mm);
  CU_TRY(cudaGetLastError());
  int h[2];
  CU_TRY(cudaMemcpyAsync(h, mm, sizeof h, cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
  if (h[0] == 0x7fffffff) return fail("dwmh_s1_minmax: the mask selects no voxel");
  for (int i = 0; i < 2; ++i) { const int o = h[i] >= 0 ? h[i] : h[i] ^ 0x7fffffff; memcpy(&out_minmax[i], &o, 4); }
  return 0;
}

extern "C" int dwmh_s1_histogram(int32_t device, const float* x, const float* mask, int64_t n, int32_t fill_outside, float fill_value,
                                 const double* edges, int32_t nbins, uint64_t* counts, void* stream_) {
  if (!x || !edges || !counts) return fail("dwmh_s1_histogram: null argument");
  if (n <= 0) return fail("dwmh_s1_histogram: empty volume");
  if (nbins < 1 || nbins > 2048) return fail("dwmh_s1_histogram: nbins = %d (1..2048 supported)", nbins);
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(device);
  CU_TRY(cudaMemsetAsync(counts, 0, (size_t)nbins * sizeof(uint64_t), st));
  const size_t smem = (size_t)(nbins + 1) * sizeof(double) + (size_t)nbins * sizeof(unsigned int);
  s1_histogram_kernel<<<sm_count(device) * 4, 256, smem, st>>>(x, mask, n, fill_outside, fill_value, edges, nbins,
                                                                 reinterpret_cast<unsigned long long*>(counts));
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_threshold_mask(int32_t device, const float* x, float threshold, const float* mul_mask, float* out, int64_t n, void* stream_) {
  if (!x || !out) return fail("dwmh_s1_threshold_mask: null argument");
  DEV_GUARD(device);
  s1_threshold_kernel<<<sm_count(device) * 8, 256, 0, (cudaStream_t)stream_>>>(x, threshold, mul_mask, out, n);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_masked_sums(int32_t device, const float* const* xs, int32_t nvol, const float* mask, int64_t n, int32_t positive_only,
                                   void* workspace, double* out_host, void* stream_) {
  if (!xs || !workspace || !out_host) return fail("dwmh_s1_masked_sums: null argument");
  if (nvol <= 0 || nvol > S1_MAX_VOLS) return fail("dwmh_s1_masked_sums: %d volumes (1..%d supported)", nvol, S1_MAX_VOLS);
  if (n <= 0) return fail("dwmh_s1_masked_sums: empty volume");
  VolPtrs vols{};
  uintptr_t al = (uintptr_t)mask;
  for (int i = 0; i < nvol; ++i) { if (!xs[i]) return fail("dwmh_s1_masked_sums: xs[%d] is null", i); vols.p[i] = const_cast<float*>(xs[i]); al |= (uintptr_t)xs[i]; }
  cudaStream_t st = (cudaStream_t)stream_;
  DEV_GUARD(device);
  double* ws = (double*)workspace;
  CU_TRY(cudaMemsetAsync(ws, 0, (size_t)nvol * ZS_SLOT * sizeof(double), st));
  CU_TRY(cudaMemset2DAsync((char*)workspace + 32, ZS_SLOT * sizeof(double), 0x7f, 4, nvol, st));
  const dim3 grid((sm_count(device) * 8 + nvol - 1) / nvol, nvol);
  if ((al & 15) == 0) s1_stats_kernel<true><<<grid, 256, 0, st>>>(vols, mask, n, ws, positive_only);
  else s1_stats_kernel<false><<<grid, 256, 0, st>>>(vols, mask, n, ws, positive_only);
  CU_TRY(cudaGetLastError());
  double h[S1_MAX_VOLS * ZS_SLOT];
  CU_TRY(cudaMemcpyAsync(h, ws, (size_t)nvol * ZS_SLOT * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
  for (int i = 0; i < nvol; ++i) for (int j = 0; j < 3; ++j) out_host[i * 3 + j] = h[i * ZS_SLOT + j];
  return 0;
}

extern "C" int dwmh_s1_label_vote(int32_t device, const float* const* labels, int32_t k, int32_t num_labels, float* averaged_label,
                                  float* tissue_majority, int64_t n, void* stream_) {
  if (!labels) return fail("dwmh_s1_label_vote: null argument");
  if (k <= 0 || k > S1_MAX_REFS) return fail("dwmh_s1_label_vote: k = %d label maps (1..%d supported)", k, S1_MAX_REFS);
  if (num_labels < 1 || num_labels > S1_MAX_LABELS) return fail("dwmh_s1_label_vote: %d label ids (1..%d supported)", num_labels, S1_MAX_LABELS);
  RefPtrs rp{};
  for (int i = 0; i < k; ++i) { if (!labels[i]) return fail("dwmh_s1_label_vote: labels[%d] is null", i); rp.p[i] = labels[i]; }
  DEV_GUARD(device);
  s1_label_vote_kernel<<<sm_count(device) * 8, 256, 0, (cudaStream_t)stream_>>>(rp, k, num_labels, averaged_label, tissue_majority, n);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_s1_apply_priors(int32_t device, float* anomaly, const float* anomaly_median, const float* averaged_label,
                                    const float* tissue_majority, int32_t stage, int64_t n, void* stream_) {
  if (!anomaly || !averaged_label) return fail("dwmh_s1_apply_priors: null argument");
  if (stage != 1 && stage != 2) return fail("dwmh_s1_apply_priors: stage must be 1 or 2");
  if (stage == 2 && (!anomaly_median || !tissue_majority)) return fail("dwmh_s1_apply_priors: stage 2 needs the median-filtered score and the tissue mask");
  DEV_GUARD(device);
  s1_apply_priors_kernel<<<sm_count(device) * 8, 256, 0, (cudaStream_t)stream_>>>(anomaly, anomaly_median, averaged_label, tissue_majority, stage, n);
  CU_TRY(cudaGetLastError());
  return 0;
}
