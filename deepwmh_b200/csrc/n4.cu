// N4 bias-field correction on the device: the `N4BiasFieldCorrection -d 3 -c [50x50x50x50,0.0] -s 2` step of
// DeepWMH_predict (deepwmh/main/predict.py:117-126), restated from Tustison et al. 2010, Sled et al. 1998 and Lee, Wolberg
// & Shin 1997 exactly as oracle/n4_oracle.py does (the [U] points are listed there and in DESIGN.md).  Fixed constants:
// 200 histogram bins, FWHM 0.15, Wiener noise 0.01, cubic B-splines on an initial 1 x 1 x 1 mesh doubled per level,
// convergence threshold 0 (every iteration runs).
//
// Shrunk points lie on a regular grid and the B-spline weights are tensor products, so the fit and the field evaluation
// are separable contractions of the [nx][ny][nz] volume with per-axis weight tables, one axis at a time.  Every output
// element is a sum in a fixed order (no floating-point atomics); the histogram accumulates fixed-point integers and the
// min / max are exact, so two calls are bit-identical.  fp64 arithmetic, fp32 storage of the two volume-sized arrays
// (log image, U = log image - field); the shrunk working set of a 182 x 218 x 182 volume (2 x 3.6 MB) stays in L2.
//
// One iteration = 6 kernels (field + min / max, histogram, sharpening table in one CTA, residual + z contraction,
// y contraction, x contraction + lattice update), captured once per level as a CUDA graph and replayed; the host
// never synchronises inside the schedule.
#include "../../include/deepwmh_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

extern "C" void dwmh_internal_set_error(const char* msg);

namespace {

int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  dwmh_internal_set_error(buf);
  return 1;
}
#define N4_CU(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) \
  return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)

struct N4DevGuard {
  int prev = -1; bool ok = false;
  explicit N4DevGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    if (prev == dev) prev = -1;
  }
  ~N4DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

constexpr int N4_BINS = 200;
constexpr int N4_PAD = 512;                          // 2^(ceil(log2 200) + 1)
constexpr int N4_OFF = (N4_PAD - N4_BINS) / 2;       // 156
constexpr double N4_FWHM = 0.15;
constexpr double N4_NOISE = 0.01;
constexpr double N4_FIX = 4294967296.0;              // histogram weights in units of 2^-32
constexpr int N4_MAX_LEVELS = 8;
constexpr int N4_MAX_ROW = 6144;                     // shrunk points per axis (one z row of fp64 per warp in shared memory)
constexpr int N4_TABLE = N4_BINS + 3;                // E[200], bin min, slope, identity flag

// Everything a kernel needs, carved out of the caller's workspace (see n4_layout).
struct N4Args {
  int nx, ny, nz;              // shrunk extents
  int X, Y, Z;                 // full-resolution extents
  int s;                       // shrink factor
  int mesh, C;                 // current level: mesh intervals per axis, control points per axis (mesh + 3)
  float* logi;                 // [nx][ny][nz] log of the shrunk image, NaN where the voxel is <= 0
  float* u;                    // [nx][ny][nz] U = logi - field
  double* t1;                  // [nx][ny][C]  after the z contraction
  double* t2;                  // [nx][C][C]   after the y contraction
  double* phi;                 // [C][C][C]    running control lattice
  double* phi_alt;             // second lattice buffer: refinement writes here, then the two swap
  double* omega;               // [C][C][C]    sum of w^2 over the valid points (per level)
  int* span[3];                // per axis and shrunk point: first control point of its span
  double* w[3];                // per axis and shrunk point: the 4 cubic weights
  double* is2[3];              // per axis and shrunk point: 1 / sum of the squared weights
  int* lo[3]; int* hi[3];      // per axis and control point: first / last shrunk point whose span covers it
  unsigned long long* hist;    // [200] fixed-point histogram
  unsigned* keys;              // [2] order-preserving keys of min / max of U over the valid points
  double* table;               // [203] sharpening table
};

__device__ __forceinline__ unsigned n4_key(float f) { const unsigned u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float n4_unkey(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// Cubic B-spline weights of full-resolution index t on the domain [0, n_full - 1] -> [0, mesh]; returns the span.
__device__ __forceinline__ int n4_bspline(int t, int n_full, int mesh, double w[4]) {
  const double u = (double)((long long)t * mesh) / (double)(n_full - 1);
  int k = (int)floor(u);
  if (k > mesh - 1) k = mesh - 1;
  const double x = u - k, y = 1.0 - x;
  w[0] = y * y * y / 6.0;
  w[1] = (3.0 * x * x * x - 6.0 * x * x + 4.0) / 6.0;
  w[2] = (-3.0 * x * x * x + 3.0 * x * x + 3.0 * x + 1.0) / 6.0;
  w[3] = x * x * x / 6.0;
  return k;
}

template <int P> __device__ __forceinline__ double n4_pow(double w) { return P == 2 ? w * w : w * w * w; }

// ---- set-up --------------------------------------------------------------------------------------------------------

// Shrink (the voxel nearest each block's centre, i * s + s / 2) and log; clears the level-0 lattice, histogram and keys.
__global__ void __launch_bounds__(256) n4_shrink_log_kernel(const float* __restrict__ in, N4Args a) {
  const int64_t n = (int64_t)a.nx * a.ny * a.nz;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int h = a.s / 2;
  for (int64_t v = g; v < n; v += stride) {
    const int k = (int)(v % a.nz), j = (int)((v / a.nz) % a.ny), i = (int)(v / ((int64_t)a.nz * a.ny));
    const float x = in[((int64_t)(i * a.s + h) * a.Y + (j * a.s + h)) * a.Z + (k * a.s + h)];
    a.logi[v] = x > 0.0f ? (float)log((double)x) : __int_as_float(0x7fc00000);
  }
  if (g < 64) a.phi[g] = 0.0;
  if (g < N4_BINS) a.hist[g] = 0ull;
  if (g == 0) { a.keys[0] = 0xffffffffu; a.keys[1] = 0u; }
}

// Per-level weight tables of the shrunk points (one CTA per axis) and, per control point, the range of points whose
// span covers it (spans grow with the index, so the range is contiguous; empty = lo > hi).
__global__ void __launch_bounds__(256) n4_tables_kernel(N4Args a) {
  const int ax = blockIdx.x;
  const int n = ax == 0 ? a.nx : (ax == 1 ? a.ny : a.nz);
  const int nf = ax == 0 ? a.X : (ax == 1 ? a.Y : a.Z);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    double w[4];
    a.span[ax][i] = n4_bspline(i * a.s + a.s / 2, nf, a.mesh, w);
    for (int q = 0; q < 4; ++q) a.w[ax][4 * i + q] = w[q];
    a.is2[ax][i] = 1.0 / (w[0] * w[0] + w[1] * w[1] + w[2] * w[2] + w[3] * w[3]);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
    int lo = n, hi = -1;
    for (int i = 0; i < n; ++i) {
      const int k = a.span[ax][i];
      if (k <= c && c <= k + 3) { lo = min(lo, i); hi = i; }
    }
    a.lo[ax][c] = lo; a.hi[ax][c] = hi;
  }
}

// Exact knot insertion (mesh -> 2 mesh) per axis: fine d = sum over coarse c of r(d - 2c + 1) phi[c], r = (1,4,6,4,1) / 8.
__device__ __forceinline__ double n4_rw(int e) {
  return e == 0 ? 0.75 : ((e == 1 || e == -1) ? 0.5 : ((e == 2 || e == -2) ? 0.125 : 0.0));
}
__global__ void __launch_bounds__(256) n4_refine_kernel(const double* __restrict__ in, int cin, double* __restrict__ out, int cout) {
  const int total = cout * cout * cout;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < total; v += gridDim.x * blockDim.x) {
    const int f = v % cout, e = (v / cout) % cout, d = v / (cout * cout);
    double acc = 0.0;
    for (int a = d / 2; a <= min(cin - 1, (d + 3) / 2); ++a) {
      const double wa = n4_rw(d - 2 * a + 1);
      for (int b = e / 2; b <= min(cin - 1, (e + 3) / 2); ++b) {
        const double wb = n4_rw(e - 2 * b + 1);
        for (int c = f / 2; c <= min(cin - 1, (f + 3) / 2); ++c)
          acc += wa * wb * n4_rw(f - 2 * c + 1) * in[(a * cin + b) * cin + c];
      }
    }
    out[v] = acc;
  }
}

// ---- one iteration -------------------------------------------------------------------------------------------------

// Field at the shrunk points, U = logi - field, exact min / max of U over the valid points.  One warp per (i, j) row:
// P[c] = sum_ab wx[a] wy[b] phi[kx + a][ky + b][c] in shared memory, then 4 taps per point along z.
__global__ void __launch_bounds__(256) n4_field_kernel(N4Args a) {
  extern __shared__ double n4_smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* P = n4_smem + wib * a.C;
  const int rows = a.nx * a.ny;
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  unsigned mn = 0xffffffffu, mx = 0u;
  for (int row = blockIdx.x * (blockDim.x >> 5) + wib; row < rows; row += nwarps) {
    const int i = row / a.ny, j = row % a.ny;
    const int kx = a.span[0][i], ky = a.span[1][j];
    const double* wx = a.w[0] + 4 * i;
    const double* wy = a.w[1] + 4 * j;
    for (int c = lane; c < a.C; c += 32) {
      double acc = 0.0;
      for (int p = 0; p < 4; ++p)
        for (int q = 0; q < 4; ++q) acc += wx[p] * wy[q] * a.phi[((kx + p) * a.C + ky + q) * a.C + c];
      P[c] = acc;
    }
    __syncwarp();
    const int64_t base = (int64_t)row * a.nz;
    for (int k = lane; k < a.nz; k += 32) {
      const int kz = a.span[2][k];
      const double* wz = a.w[2] + 4 * k;
      const double b = wz[0] * P[kz] + wz[1] * P[kz + 1] + wz[2] * P[kz + 2] + wz[3] * P[kz + 3];
      const float l = a.logi[base + k];
      const float uv = (float)((double)l - b);               // NaN stays NaN
      a.u[base + k] = uv;
      if (!isnan(uv)) { const unsigned key = n4_key(uv); mn = min(mn, key); mx = max(mx, key); }
    }
    __syncwarp();
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
  __shared__ unsigned smn[8], smx[8];
  if (lane == 0) { smn[wib] = mn; smx[wib] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { mn = min(mn, smn[w]); mx = max(mx, smx[w]); }
    if (mn <= mx) { atomicMin(a.keys, mn); atomicMax(a.keys + 1, mx); }
  }
}

// 200-bin histogram of U with linear splatting; weights are fixed-point integers, so the sums do not depend on order.
__global__ void __launch_bounds__(256) n4_hist_kernel(N4Args a) {
  __shared__ unsigned long long sh[N4_BINS];
  for (int b = threadIdx.x; b < N4_BINS; b += blockDim.x) sh[b] = 0ull;
  __syncthreads();
  const double lo = (double)n4_unkey(a.keys[0]), hi = (double)n4_unkey(a.keys[1]);
  const double slope = (hi - lo) / (N4_BINS - 1);
  if (a.keys[0] <= a.keys[1] && slope > 0.0) {
    const int64_t n = (int64_t)a.nx * a.ny * a.nz;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x) {
      const float uv = a.u[v];
      if (isnan(uv)) continue;
      const double cidx = ((double)uv - lo) / slope;
      const int idx = min((int)floor(cidx), N4_BINS - 1);
      const unsigned long long wh = idx == N4_BINS - 1 ? 0ull : (unsigned long long)rint((cidx - idx) * N4_FIX);
      atomicAdd(&sh[idx], (unsigned long long)N4_FIX - wh);
      if (wh) atomicAdd(&sh[idx + 1], wh);
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < N4_BINS; b += blockDim.x)
    if (sh[b]) atomicAdd(a.hist + b, sh[b]);
}

// In-place radix-2 FFT of 512 complex points in shared memory by the 256 threads tid = 0 .. 255 (decimation in time after
// the bit-reversal permutation), unnormalised; sign -1: forward (numpy.fft.fft), +1: inverse without the 1 / 512.
// Every thread of the block calls it (it contains __syncthreads); threads with active == false only keep step.
__device__ void n4_fft512(double* re, double* im, const double* twc, const double* tws, double sign, int tid, bool active) {
  if (active) {
    for (int i = tid; i < N4_PAD; i += 256) {
      const int j = (int)(__brev((unsigned)i) >> 23);
      if (j > i) { const double r = re[i], m = im[i]; re[i] = re[j]; im[i] = im[j]; re[j] = r; im[j] = m; }
    }
  }
  __syncthreads();
  for (int len = 2; len <= N4_PAD; len <<= 1) {
    if (active) {
      const int half = len >> 1, pos = tid & (half - 1);
      const int i0 = (tid - pos) * 2 + pos, i1 = i0 + half;
      const int tw = pos * (N4_PAD / len);
      const double wr = twc[tw], wi = sign * tws[tw];
      const double xr = re[i1] * wr - im[i1] * wi, xi = re[i1] * wi + im[i1] * wr;
      re[i1] = re[i0] - xr; im[i1] = im[i0] - xi;
      re[i0] += xr; im[i0] += xi;
    }
    __syncthreads();
  }
}

// Sharpening table (one CTA of 512 threads, fp64), ITK's FFT formulation: Wiener deconvolution of the padded histogram V by
// the circular Gaussian F of FWHM 0.15 / slope bins (U = IFFT(FFT(V) conj(F^) / (|F^|^2 + noise)), clamped at 0), then
// E[u | u^] = IFFT(FFT(centre U) F^) / IFFT(FFT(U) F^) at the 200 bins (a common scale of U cancels in the ratio).
// The two halves of the block transform two arrays at once.  Resets histogram and keys for the next iteration.
__global__ void __launch_bounds__(N4_PAD) n4_sharpen_kernel(N4Args a) {
  __shared__ double twc[N4_PAD / 2], tws[N4_PAD / 2];
  __shared__ double fr[N4_PAD], fi[N4_PAD], br[N4_PAD], bi[N4_PAD], cr[N4_PAD], ci[N4_PAD];
  const int t = threadIdx.x, tid = t & 255;
  const bool upper = t >= 256;
  const unsigned k0 = a.keys[0], k1 = a.keys[1];
  const double lo = (double)n4_unkey(k0), hi = (double)n4_unkey(k1);
  const double slope = (hi - lo) / (N4_BINS - 1);
  const bool identity = !(k0 <= k1) || !(slope > 0.0);
  const double sfwhm = N4_FWHM / slope;
  const double expf_ = 4.0 * log(2.0) / (sfwhm * sfwhm);
  const double scale = 2.0 * sqrt(log(2.0) / M_PI) / sfwhm;
  const int m = min(t, N4_PAD - t);
  if (t < N4_PAD / 2) { twc[t] = cospi((double)t / (N4_PAD / 2)); tws[t] = sinpi((double)t / (N4_PAD / 2)); }
  fr[t] = t == 0 ? scale : scale * exp(-(double)m * m * expf_); fi[t] = 0.0;
  br[t] = (t >= N4_OFF && t < N4_OFF + N4_BINS) ? (double)a.hist[t - N4_OFF] / N4_FIX : 0.0; bi[t] = 0.0;
  __syncthreads();
  n4_fft512(upper ? br : fr, upper ? bi : fi, twc, tws, -1.0, tid, true);              // F^, V^
  {
    const double den = fr[t] * fr[t] + fi[t] * fi[t] + N4_NOISE;
    const double gr = fr[t] / den, gi = -fi[t] / den;
    cr[t] = br[t] * gr - bi[t] * gi; ci[t] = br[t] * gi + bi[t] * gr;
  }
  __syncthreads();
  n4_fft512(cr, ci, twc, tws, 1.0, tid, !upper);                                         // U (times 512)
  const double u = fmax(cr[t], 0.0);
  __syncthreads();
  br[t] = (lo + (double)(t - N4_OFF) * slope) * u; bi[t] = 0.0;
  cr[t] = u; ci[t] = 0.0;
  __syncthreads();
  n4_fft512(upper ? cr : br, upper ? ci : bi, twc, tws, -1.0, tid, true);
  {
    const double xr = br[t], xi = bi[t], yr = cr[t], yi = ci[t];
    br[t] = xr * fr[t] - xi * fi[t]; bi[t] = xr * fi[t] + xi * fr[t];
    cr[t] = yr * fr[t] - yi * fi[t]; ci[t] = yr * fi[t] + yi * fr[t];
  }
  __syncthreads();
  n4_fft512(upper ? cr : br, upper ? ci : bi, twc, tws, 1.0, tid, true);
  if (t >= N4_OFF && t < N4_OFF + N4_BINS) {
    const double nu = br[t], de = cr[t];
    a.table[t - N4_OFF] = de != 0.0 ? nu / de : 0.0;
  }
  if (t == 0) { a.table[N4_BINS] = lo; a.table[N4_BINS + 1] = slope; a.table[N4_BINS + 2] = identity ? 1.0 : 0.0; }
  if (t < N4_BINS) a.hist[t] = 0ull;
  if (t == 0) { a.keys[0] = 0xffffffffu; a.keys[1] = 0u; }
}

__device__ __forceinline__ double n4_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Residual (MODE 0: R = U - sharpened(U), scaled by 1 / sum w^2 = 1 / (Sx Sy Sz), weights w^3) or validity (MODE 1:
// weights w^2, for omega) of one (i, j) row into shared memory, then its z contraction t1[i][j][c]: one warp per row,
// the lanes split the points of each control point's range and a fixed shuffle tree adds them.
template <int MODE>
__global__ void __launch_bounds__(256) n4_residual_z_kernel(N4Args a) {
  extern __shared__ double n4_smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* r = n4_smem + (int64_t)wib * a.nz;
  const int rows = a.nx * a.ny;
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  const double* E = a.table;
  const double lo = E[N4_BINS], slope = E[N4_BINS + 1];
  const bool identity = E[N4_BINS + 2] != 0.0;
  for (int row = blockIdx.x * (blockDim.x >> 5) + wib; row < rows; row += nwarps) {
    const int i = row / a.ny, j = row % a.ny;
    const int64_t base = (int64_t)row * a.nz;
    const double isxy = a.is2[0][i] * a.is2[1][j];
    for (int k = lane; k < a.nz; k += 32) {
      double v = 0.0;
      if (MODE == 1) {
        v = isnan(a.logi[base + k]) ? 0.0 : 1.0;
      } else {
        const float uv = a.u[base + k];
        if (!isnan(uv) && !identity) {
          const double x = (double)uv;
          const double cidx = (x - lo) / slope;
          const int idx = (int)floor(cidx);
          const double sh = idx < N4_BINS - 1 ? E[idx] + (E[idx + 1] - E[idx]) * (cidx - idx) : E[N4_BINS - 1];
          v = (x - sh) * (isxy * a.is2[2][k]);
        }
      }
      r[k] = v;
    }
    __syncwarp();
    for (int c = 0; c < a.C; ++c) {
      double acc = 0.0;
      for (int k = a.lo[2][c] + lane; k <= a.hi[2][c]; k += 32)
        acc += n4_pow<MODE == 0 ? 3 : 2>(a.w[2][4 * k + (c - a.span[2][k])]) * r[k];
      acc = n4_warp_sum(acc);
      if (lane == 0) a.t1[(int64_t)row * a.C + c] = acc;
    }
    __syncwarp();
  }
}

// y contraction: t2[i][b][c] = sum_j wy(j)[b]^P t1[i][j][c], one warp per output.
template <int P>
__global__ void __launch_bounds__(256, 2) n4_contract_y_kernel(N4Args a) {
  const int lane = threadIdx.x & 31;
  const int total = a.nx * a.C * a.C;
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  for (int v = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); v < total; v += nwarps) {
    const int c = v % a.C, b = (v / a.C) % a.C, i = v / (a.C * a.C);
    double acc = 0.0;
    for (int j = a.lo[1][b] + lane; j <= a.hi[1][b]; j += 32)
      acc += n4_pow<P>(a.w[1][4 * j + (b - a.span[1][j])]) * a.t1[((int64_t)i * a.ny + j) * a.C + c];
    acc = n4_warp_sum(acc);
    if (lane == 0) a.t2[v] = acc;
  }
}

// x contraction and the lattice update, one warp per output: delta[a][b][c] = sum_i wx(i)[a]^P t2[i][b][c];
// MODE 0: phi += delta / omega (0 where omega is 0), MODE 1: omega = delta.
template <int MODE>
__global__ void __launch_bounds__(256) n4_contract_x_kernel(N4Args a) {
  const int lane = threadIdx.x & 31;
  const int total = a.C * a.C * a.C;
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  for (int v = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); v < total; v += nwarps) {
    const int bc = v % (a.C * a.C), p = v / (a.C * a.C);
    double acc = 0.0;
    for (int i = a.lo[0][p] + lane; i <= a.hi[0][p]; i += 32)
      acc += n4_pow<MODE == 0 ? 3 : 2>(a.w[0][4 * i + (p - a.span[0][i])]) * a.t2[(int64_t)i * a.C * a.C + bc];
    acc = n4_warp_sum(acc);
    if (lane == 0) {
      if (MODE == 1) a.omega[v] = acc;
      else { const double om = a.omega[v]; if (om > 0.0) a.phi[v] += acc / om; }
    }
  }
}

// ---- output --------------------------------------------------------------------------------------------------------

// Field at every full-resolution voxel, out = in / exp(field), log_field = field.  One warp per (x, y) row; in may alias out.
__global__ void __launch_bounds__(256) n4_output_kernel(const float* in, float* out, float* __restrict__ log_field, N4Args a) {
  extern __shared__ double n4_smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* P = n4_smem + wib * a.C;
  const int rows = a.X * a.Y;
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  for (int row = blockIdx.x * (blockDim.x >> 5) + wib; row < rows; row += nwarps) {
    const int x = row / a.Y, y = row % a.Y;
    double wx[4], wy[4];
    const int kx = n4_bspline(x, a.X, a.mesh, wx), ky = n4_bspline(y, a.Y, a.mesh, wy);
    for (int c = lane; c < a.C; c += 32) {
      double acc = 0.0;
      for (int p = 0; p < 4; ++p)
        for (int q = 0; q < 4; ++q) acc += wx[p] * wy[q] * a.phi[((kx + p) * a.C + ky + q) * a.C + c];
      P[c] = acc;
    }
    __syncwarp();
    const int64_t base = (int64_t)row * a.Z;
    for (int z = lane; z < a.Z; z += 32) {
      double wz[4];
      const int kz = n4_bspline(z, a.Z, a.mesh, wz);
      const double b = wz[0] * P[kz] + wz[1] * P[kz + 1] + wz[2] * P[kz + 2] + wz[3] * P[kz + 3];
      const float v = in[base + z];
      out[base + z] = (float)((double)v / exp(b));
      if (log_field) log_field[base + z] = (float)b;
    }
    __syncwarp();
  }
}

// ---- host ----------------------------------------------------------------------------------------------------------

int64_t align256(int64_t b) { return (b + 255) / 256 * 256; }

// Workspace layout; with base == nullptr only the total is computed.
int64_t n4_layout(int X, int Y, int Z, int s, int levels, char* base, N4Args* a) {
  const int nx = X / s, ny = Y / s, nz = Z / s;
  const int cmax = (1 << (levels - 1)) + 3;
  const int64_t n = (int64_t)nx * ny * nz;
  int64_t off = 0;
  auto take = [&](int64_t bytes) { char* p = base ? base + off : nullptr; off += align256(bytes); return p; };
  N4Args t{};
  t.logi = (float*)take(n * 4);
  t.u = (float*)take(n * 4);
  t.t1 = (double*)take((int64_t)nx * ny * cmax * 8);
  t.t2 = (double*)take((int64_t)nx * cmax * cmax * 8);
  t.phi = (double*)take((int64_t)cmax * cmax * cmax * 8);
  t.phi_alt = (double*)take((int64_t)cmax * cmax * cmax * 8);
  t.omega = (double*)take((int64_t)cmax * cmax * cmax * 8);
  const int ext[3] = {nx, ny, nz};
  for (int ax = 0; ax < 3; ++ax) {
    t.span[ax] = (int*)take((int64_t)ext[ax] * 4);
    t.w[ax] = (double*)take((int64_t)ext[ax] * 32);
    t.is2[ax] = (double*)take((int64_t)ext[ax] * 8);
    t.lo[ax] = (int*)take((int64_t)cmax * 4);
    t.hi[ax] = (int*)take((int64_t)cmax * 4);
  }
  t.hist = (unsigned long long*)take(N4_BINS * 8);
  t.keys = (unsigned*)take(8);
  t.table = (double*)take(N4_TABLE * 8);
  if (a) {
    *a = t;
    a->nx = nx; a->ny = ny; a->nz = nz; a->X = X; a->Y = Y; a->Z = Z; a->s = s;
  }
  return off;
}

int n4_check(int X, int Y, int Z, int s, int levels) {
  if (X <= 0 || Y <= 0 || Z <= 0) return fail("dwmh_n4: empty extent %d x %d x %d", X, Y, Z);
  if (s < 1) return fail("dwmh_n4: shrink factor %d (>= 1)", s);
  if (levels < 1 || levels > N4_MAX_LEVELS) return fail("dwmh_n4: %d fitting levels (1 .. %d)", levels, N4_MAX_LEVELS);
  const int e[3] = {X / s, Y / s, Z / s};
  for (int ax = 0; ax < 3; ++ax) {
    if (e[ax] < 2) return fail("dwmh_n4: shrink factor %d leaves %d point(s) on axis %d of %d x %d x %d (>= 2 needed)", s, e[ax], ax, X, Y, Z);
    if (e[ax] > N4_MAX_ROW) return fail("dwmh_n4: %d shrunk points on axis %d (<= %d)", e[ax], ax, N4_MAX_ROW);
  }
  return 0;
}

// Blocks of 8 warps for `outputs` warp-per-output items, at most `grid`.
int n4_warp_grid(int outputs, int grid) { return std::max(1, std::min(grid, (outputs + 7) / 8)); }

// The six kernels of one iteration, in order, on `st`.
void n4_iteration(const N4Args& a, int grid, int warps_z, cudaStream_t st) {
  const size_t smem_c = (size_t)8 * a.C * sizeof(double);
  n4_field_kernel<<<grid, 256, smem_c, st>>>(a);
  n4_hist_kernel<<<grid, 256, 0, st>>>(a);
  n4_sharpen_kernel<<<1, N4_PAD, 0, st>>>(a);
  n4_residual_z_kernel<0><<<grid, warps_z * 32, (size_t)warps_z * a.nz * sizeof(double), st>>>(a);
  n4_contract_y_kernel<3><<<n4_warp_grid(a.nx * a.C * a.C, grid), 256, 0, st>>>(a);
  n4_contract_x_kernel<0><<<n4_warp_grid(a.C * a.C * a.C, grid), 256, 0, st>>>(a);
}

}  // namespace

extern "C" int dwmh_n4_workspace(int32_t X, int32_t Y, int32_t Z, int32_t shrink, int32_t num_levels, int64_t* bytes) {
  if (!bytes) return fail("dwmh_n4_workspace: null argument");
  if (n4_check(X, Y, Z, shrink, num_levels)) return 1;
  *bytes = n4_layout(X, Y, Z, shrink, num_levels, nullptr, nullptr);
  return 0;
}

extern "C" int dwmh_n4(int32_t device, const float* in, int32_t X, int32_t Y, int32_t Z, int32_t shrink, int32_t num_levels,
                       const int32_t* iterations, float* out, float* log_field, void* workspace, void* stream_) {
  if (!in || !out || !iterations || !workspace) return fail("dwmh_n4: null argument");
  if (n4_check(X, Y, Z, shrink, num_levels)) return 1;
  for (int l = 0; l < num_levels; ++l)
    if (iterations[l] < 0) return fail("dwmh_n4: %d iterations on level %d", iterations[l], l);
  N4DevGuard dg(device);
  if (!dg.ok) return fail("cudaSetDevice(%d) failed", device);
  cudaStream_t st = (cudaStream_t)stream_;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const int grid = sms * 4;
  N4Args a;
  n4_layout(X, Y, Z, shrink, num_levels, (char*)workspace, &a);
  const int warps_z = std::max(1, std::min(8, (48 * 1024) / (a.nz * (int)sizeof(double))));

  a.mesh = 1; a.C = 4;
  n4_shrink_log_kernel<<<grid, 256, 0, st>>>(in, a);
  N4_CU(cudaGetLastError());
  cudaStream_t cs = nullptr;                 // private stream, used only to capture the per-level graph
  N4_CU(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  int rc = 0;
  for (int level = 0; level < num_levels && rc == 0; ++level) {
    if (level > 0) {
      const int cin = a.C;
      a.mesh *= 2; a.C = a.mesh + 3;
      n4_refine_kernel<<<std::max(1, std::min(grid, (a.C * a.C * a.C + 255) / 256)), 256, 0, st>>>(a.phi, cin, a.phi_alt, a.C);
      std::swap(a.phi, a.phi_alt);
    }
    n4_tables_kernel<<<3, 256, 0, st>>>(a);
    n4_residual_z_kernel<1><<<grid, warps_z * 32, (size_t)warps_z * a.nz * sizeof(double), st>>>(a);
    n4_contract_y_kernel<2><<<n4_warp_grid(a.nx * a.C * a.C, grid), 256, 0, st>>>(a);
    n4_contract_x_kernel<1><<<n4_warp_grid(a.C * a.C * a.C, grid), 256, 0, st>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { rc = fail("dwmh_n4: level %d set-up launch failed: %s", level, cudaGetErrorString(e)); break; }
    if (iterations[level] == 0) continue;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
    if (e == cudaSuccess) {
      n4_iteration(a, grid, warps_z, cs);
      const cudaError_t el = cudaGetLastError();
      e = cudaStreamEndCapture(cs, &graph);
      if (e == cudaSuccess) e = el;
    }
    if (e == cudaSuccess) e = cudaGraphInstantiate(&exec, graph, 0);
    for (int it = 0; e == cudaSuccess && it < iterations[level]; ++it) e = cudaGraphLaunch(exec, st);
    if (exec) cudaGraphExecDestroy(exec);  // in-flight launches complete before the graph is freed
    if (graph) cudaGraphDestroy(graph);
    if (e != cudaSuccess) rc = fail("dwmh_n4: level %d iteration graph failed: %s", level, cudaGetErrorString(e));
  }
  cudaStreamDestroy(cs);
  if (rc) return rc;
  n4_output_kernel<<<grid, 256, (size_t)8 * a.C * sizeof(double), st>>>(in, out, log_field, a);
  N4_CU(cudaGetLastError());
  return 0;
}
