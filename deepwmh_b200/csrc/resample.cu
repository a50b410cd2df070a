// Spacing resample of SURVEY.md section 8f-1 on the device: what nnU-Net v1 does to every case whose voxel spacing differs
// from the plans' (resample_patient / resample_data_or_seg [U:preprocessing/preprocessing.py], the resample-back of
// save_segmentation_nifti_from_softmax [U:inference/segmentation_export.py]; reached from deepwmh/main/predict.py:153-156).
// The arithmetic upstream delegates to is skimage.transform.resize(order, mode='edge', anti_aliasing=False, clip=True), i.e.
// scipy.ndimage.zoom(order, mode='nearest', grid_mode=True) + clip, all in float64:
//   order 3: edge-pad by 12, cubic B-spline prefilter (pole sqrt(3) - 2, mirror boundaries on the padded array) per axis,
//            then 4 x 4 x 4 B-spline taps at (o + 0.5) * n_in / n_out - 0.5;
//   order 1: 2 x 2 x 2 linear taps at the same coordinates clamped to [0, n - 1];
//   separate-z (anisotropy > 3): the resize runs per slice in-plane, the coarse axis is nearest-neighbour
//            (map_coordinates order 0: floor(c + 0.5) of the clamped coordinate); the clip range is then per source slice.
// HBM-bound gather kernels (coalesced along z, grid = multiple of the SM count); the prefilter is a 49-tap FIR with the
// exact impulse response sqrt(3) * z^|k| (|z|^24 = 2e-14) instead of the recursive filter, which does not parallelise.
// Context-free entry points (no network involved), as the stage-1 ones.
#include "../../include/deepwmh_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cuda_runtime.h>

#include "host.cuh"
#include "common.cuh"

using dwmh::fail;
using dwmh::sm_count;

namespace {

using dwmh::float_key;
using dwmh::key_float;

constexpr int RS_NPAD = 12;        // scipy's _prepad_for_spline_filter for mode 'nearest'
constexpr int RS_RADIUS = 24;      // FIR radius of the prefilter
constexpr int RS_MARGIN = 2;       // coefficients kept beyond either end of a cubic axis (taps floor(c) - 1 .. floor(c) + 2)

__constant__ double c_fir[RS_RADIUS + 1];      // sqrt(3) * z^k

// signal extension scipy applies before / inside the prefilter: edge-replicate 12 samples, mirror beyond
__device__ __forceinline__ int rs_ext(int i, int n) {
  int p = i + RS_NPAD;
  const int N = n + 2 * RS_NPAD;
  if (p < 0) p = -p;
  if (p > N - 1) p = 2 * (N - 1) - p;
  p -= RS_NPAD;
  return p < 0 ? 0 : (p > n - 1 ? n - 1 : p);
}

// min / max of every slice along `axis` (axis < 0: the whole volume is one slice): grid (nslices, chunks); a block reduces its
// share of one slice and issues one atomicMin / atomicMax.  range[2 s] = min key, range[2 s + 1] = max key.
__global__ void __launch_bounds__(256) rs_range_kernel(const float* __restrict__ src, int n0, int n1, int n2, int axis, unsigned* __restrict__ range) {
  const int s = blockIdx.x;
  const int64_t M = axis < 0 ? (int64_t)n0 * n1 * n2 : (axis == 0 ? (int64_t)n1 * n2 : (axis == 1 ? (int64_t)n0 * n2 : (int64_t)n0 * n1));
  unsigned mn = 0xffffffffu, mx = 0u;
  for (int64_t e = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; e < M; e += (int64_t)gridDim.y * blockDim.x) {
    int64_t idx;
    if (axis <= 0) idx = (int64_t)s * M + e;                                  // axis 0 (or whole volume, s = 0): contiguous
    else if (axis == 1) idx = ((e / n2) * n1 + s) * n2 + e % n2;              // (i0, i2) with i2 fastest
    else idx = e * n2 + s;                                                    // (i0, i1), strided
    const unsigned k = float_key(src[idx]);
    mn = min(mn, k); mx = max(mx, k);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
  __shared__ unsigned smn[8], smx[8];
  if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { mn = min(mn, smn[w]); mx = max(mx, smx[w]); }
    atomicMin(range + 2 * s, mn); atomicMax(range + 2 * s + 1, mx);
  }
}

__global__ void rs_range_init_kernel(unsigned* range, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { range[2 * i] = 0xffffffffu; range[2 * i + 1] = 0u; }
}

// One prefilter pass along `axis`: out has the input's extents except along `axis`, where it covers [-MARGIN, n + MARGIN).
// TIn = float (first pass, reads the source volume) or double.
template <typename TIn>
__global__ void __launch_bounds__(256) rs_prefilter_kernel(const TIn* __restrict__ in, double* __restrict__ out, int d0, int d1, int d2, int axis) {
  // (d0, d1, d2) = extents of `in`
  const int o0 = d0 + (axis == 0 ? 2 * RS_MARGIN : 0), o1 = d1 + (axis == 1 ? 2 * RS_MARGIN : 0), o2 = d2 + (axis == 2 ? 2 * RS_MARGIN : 0);
  const int64_t V = (int64_t)o0 * o1 * o2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int n = axis == 0 ? d0 : (axis == 1 ? d1 : d2);
  const int64_t astride = axis == 0 ? (int64_t)d1 * d2 : (axis == 1 ? d2 : 1);
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += stride) {
    int i2 = (int)(v % o2), i1 = (int)((v / o2) % o1), i0 = (int)(v / ((int64_t)o2 * o1));
    int c = (axis == 0 ? i0 : (axis == 1 ? i1 : i2)) - RS_MARGIN;          // position along the filtered axis
    if (axis == 0) i0 = 0; else if (axis == 1) i1 = 0; else i2 = 0;
    const TIn* base = in + ((int64_t)i0 * d1 + i1) * d2 + i2;
    double acc = c_fir[0] * (double)base[(int64_t)rs_ext(c, n) * astride];
    for (int k = 1; k <= RS_RADIUS; ++k)
      acc += c_fir[k] * ((double)base[(int64_t)rs_ext(c - k, n) * astride] + (double)base[(int64_t)rs_ext(c + k, n) * astride]);
    out[v] = acc;
  }
}

__global__ void __launch_bounds__(256) rs_to_double_kernel(const float* __restrict__ in, double* __restrict__ out, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = (double)in[i];
}

struct RsAxis {
  int mode;        // 0 nearest (order 0), 1 linear, 3 cubic
  int n_in, n_out;
  int margin;      // RS_MARGIN for a cubic axis (the coefficient array is extended), else 0
  double scale;    // n_in / n_out
};
struct RsParams { RsAxis ax[3]; int clip_axis; int out_mode; };

// taps of one axis at output index o: first source index (in the extended array) and up to 4 weights, scipy's formulas
__device__ __forceinline__ int rs_taps(const RsAxis& a, int o, int& base, double w[4], int& slice) {
  double cc = __dsub_rn(__dmul_rn((double)o + 0.5, a.scale), 0.5);      // two roundings, as the C reference evaluates it (no FMA)
  if (a.mode == 3) {
    const double fl = floor(cc);
    const double y = cc - fl, z = 1.0 - y;
    w[1] = (y * y * (y - 2.0) * 3.0 + 4.0) / 6.0;
    w[2] = (z * z * (z - 2.0) * 3.0 + 4.0) / 6.0;
    w[0] = z * z * z / 6.0;
    w[3] = 1.0 - w[0] - w[1] - w[2];
    base = (int)fl - 1 + a.margin;
    slice = 0;
    return 4;
  }
  cc = cc < 0.0 ? 0.0 : (cc > (double)(a.n_in - 1) ? (double)(a.n_in - 1) : cc);      // map_coordinate, mode 'nearest'
  if (a.mode == 1) {
    const double fl = floor(cc);
    const double y = cc - fl;
    w[0] = 1.0 - y; w[1] = y;
    base = (int)fl;
    slice = 0;
    return 2;
  }
  base = (int)floor(cc + 0.5);
  if (base > a.n_in - 1) base = a.n_in - 1;
  w[0] = 1.0;
  slice = base;
  return 1;
}

// out[o0][o1][o2] = sum over taps of coef * w0 * w1 * w2 in scipy's evaluation order (no FMA contraction), clipped to the
// range of the source (slice), cast to fp32 -- or thresholded to nnU-Net's crop-mask labels (>= 0.5 ? 0 : -1).
__global__ void __launch_bounds__(256) rs_gather_kernel(const double* __restrict__ coef, void* __restrict__ out, RsParams p,
                                                        const unsigned* __restrict__ range) {
  const int O0 = p.ax[0].n_out, O1 = p.ax[1].n_out, O2 = p.ax[2].n_out;
  const int E1 = p.ax[1].n_in + 2 * p.ax[1].margin, E2 = p.ax[2].n_in + 2 * p.ax[2].margin;
  const int L0 = p.ax[0].n_in + 2 * p.ax[0].margin - 1, L1 = E1 - 1, L2 = E2 - 1;
  const int64_t V = (int64_t)O0 * O1 * O2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += stride) {
    const int o2 = (int)(v % O2), o1 = (int)((v / O2) % O1), o0 = (int)(v / ((int64_t)O2 * O1));
    int b0, b1, b2, s0, s1, s2;
    double w0[4], w1[4], w2[4];
    const int t0 = rs_taps(p.ax[0], o0, b0, w0, s0), t1 = rs_taps(p.ax[1], o1, b1, w1, s1), t2 = rs_taps(p.ax[2], o2, b2, w2, s2);
    double t = 0.0;
    for (int a = 0; a < t0; ++a) {
      const int i0 = min(max(b0 + a, 0), L0);
      for (int b = 0; b < t1; ++b) {
        const int i1 = min(max(b1 + b, 0), L1);
        const double* row = coef + ((int64_t)i0 * E1 + i1) * E2;
        for (int c = 0; c < t2; ++c) {
          const int i2 = min(max(b2 + c, 0), L2);
          const double x = __dmul_rn(__dmul_rn(__dmul_rn(row[i2], w0[a]), w1[b]), w2[c]);
          t = __dadd_rn(t, x);
        }
      }
    }
    const int s = p.clip_axis < 0 ? 0 : (p.clip_axis == 0 ? s0 : (p.clip_axis == 1 ? s1 : s2));
    const double lo = (double)key_float(range[2 * s]), hi = (double)key_float(range[2 * s + 1]);
    t = t < lo ? lo : (t > hi ? hi : t);
    if (p.out_mode == 1) reinterpret_cast<int8_t*>(out)[v] = t >= 0.5 ? 0 : -1;
    else reinterpret_cast<float*>(out)[v] = (float)t;
  }
}

// The cascade's previous-stage input [U:predict.py::preprocess_save_to_queue]: resize_segmentation(labels, out shape,
// order 1) then one-hot over classes 1 .. C-1, written straight into C-1 fp32 planes of the network input.  Per voxel and
// class c (ascending), the order-1 resize of the 0/1 indicator of c is rs_gather_kernel's sum over the 2 x 2 x 2 taps of
// rs_taps; a tap of value 0 adds an exact 0 and a tap of value 1 adds w0 * w1 * w2, so only the taps holding c are added,
// in the same order.  Where that sum is >= 0.5, c is written (later classes overwrite earlier ones).  The clip to the
// indicator's range cannot move a sum across 0.5, so it is left out.
__global__ void __launch_bounds__(256) rs_onehot_kernel(const uint8_t* __restrict__ labels, float* __restrict__ dst, RsParams p,
                                                        int num_classes) {
  const int N0 = p.ax[0].n_in, N1 = p.ax[1].n_in, N2 = p.ax[2].n_in;
  const int O0 = p.ax[0].n_out, O1 = p.ax[1].n_out, O2 = p.ax[2].n_out;
  const int64_t V = (int64_t)O0 * O1 * O2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += stride) {
    const int o2 = (int)(v % O2), o1 = (int)((v / O2) % O1), o0 = (int)(v / ((int64_t)O2 * O1));
    int b0, b1, b2, s0, s1, s2;
    double w0[4], w1[4], w2[4];
    rs_taps(p.ax[0], o0, b0, w0, s0); rs_taps(p.ax[1], o1, b1, w1, s1); rs_taps(p.ax[2], o2, b2, w2, s2);
    uint8_t lab[2][2][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b)
#pragma unroll
        for (int c = 0; c < 2; ++c)
          lab[a][b][c] = labels[((int64_t)min(b0 + a, N0 - 1) * N1 + min(b1 + b, N1 - 1)) * N2 + min(b2 + c, N2 - 1)];
    int out = 0;
    for (int k = 1; k < num_classes; ++k) {
      double t = 0.0;
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b)
#pragma unroll
          for (int c = 0; c < 2; ++c)
            if (lab[a][b][c] == k) t = __dadd_rn(t, __dmul_rn(__dmul_rn(w0[a], w1[b]), w2[c]));
      if (t >= 0.5) out = k;
    }
    for (int k = 1; k < num_classes; ++k) dst[(size_t)(k - 1) * V + v] = out == k ? 1.f : 0.f;
  }
}

bool fir_ready[64] = {false};

}  // namespace

static int64_t rs_ws_doubles(const int32_t in_shape[3], int32_t order, int32_t separate_axis) {
  int64_t v = 1;
  for (int a = 0; a < 3; ++a) v *= in_shape[a] + ((order == 3 && a != separate_axis) ? 2 * RS_MARGIN : 0);
  return v;
}

extern "C" int dwmh_resample_workspace(const int32_t in_shape[3], int32_t order, int32_t separate_axis, int64_t* bytes) {
  if (!in_shape || !bytes) return fail("dwmh_resample_workspace: null argument");
  const int64_t slices = separate_axis >= 0 ? in_shape[separate_axis] : 1;
  // two ping-pong coefficient arrays in fp64 + the clip ranges
  *bytes = 2 * rs_ws_doubles(in_shape, order, separate_axis) * (int64_t)sizeof(double) + (2 * slices * (int64_t)sizeof(unsigned) + 255) / 256 * 256;
  return 0;
}

extern "C" int dwmh_resample(int32_t device, const float* src, const int32_t in_shape[3], void* dst, const int32_t out_shape[3],
                             int32_t order, int32_t separate_axis, int32_t out_mode, void* workspace, void* stream_) {
  if (!src || !dst || !in_shape || !out_shape || !workspace) return fail("dwmh_resample: null argument");
  if (order != 0 && order != 1 && order != 3) return fail("dwmh_resample: order %d (0, 1 or 3; nnU-Net uses 3 for data, 1 for masks / softmax)", order);
  if (separate_axis < -1 || separate_axis > 2) return fail("dwmh_resample: separate_axis %d", separate_axis);
  if (out_mode != 0 && out_mode != 1) return fail("dwmh_resample: out_mode %d", out_mode);
  for (int a = 0; a < 3; ++a)
    if (in_shape[a] <= 0 || out_shape[a] <= 0) return fail("dwmh_resample: empty extent on axis %d", a);
  DEV_GUARD(device);
  cudaStream_t st = (cudaStream_t)stream_;
  if (device >= 0 && device < 64 && !fir_ready[device]) {
    double h[RS_RADIUS + 1];
    const double z = std::sqrt(3.0) - 2.0;
    double zk = 1.0;
    for (int k = 0; k <= RS_RADIUS; ++k) { h[k] = std::sqrt(3.0) * zk; zk *= z; }
    CU_TRY(cudaMemcpyToSymbol(c_fir, h, sizeof h));
    fir_ready[device] = true;
  }
  const int grid = sm_count(device) * 8;
  const int64_t wsd = rs_ws_doubles(in_shape, order, separate_axis);
  double* bufA = reinterpret_cast<double*>(workspace);
  double* bufB = bufA + wsd;
  unsigned* range = reinterpret_cast<unsigned*>(bufB + wsd);
  const int nslices = separate_axis >= 0 ? in_shape[separate_axis] : 1;
  rs_range_init_kernel<<<(nslices + 255) / 256, 256, 0, st>>>(range, nslices);
  {
    const int chunks = std::max(1, std::min(grid / nslices, 1024));
    rs_range_kernel<<<dim3(nslices, chunks), 256, 0, st>>>(src, in_shape[0], in_shape[1], in_shape[2], separate_axis, range);
  }
  // coefficient array (fp64): prefiltered along the cubic axes (z, y, x in turn), a plain conversion otherwise
  int d[3] = {in_shape[0], in_shape[1], in_shape[2]};
  const double* coef = nullptr;
  bool first = true;
  double* cur = bufA; double* nxt = bufB;
  if (order == 3) {
    for (int axis = 2; axis >= 0; --axis) {
      if (axis == separate_axis) continue;
      if (first) rs_prefilter_kernel<float><<<grid, 256, 0, st>>>(src, cur, d[0], d[1], d[2], axis);
      else { rs_prefilter_kernel<double><<<grid, 256, 0, st>>>(coef, nxt, d[0], d[1], d[2], axis); std::swap(cur, nxt); }
      coef = cur;
      d[axis] += 2 * RS_MARGIN;
      first = false;
    }
  }
  if (!coef) {
    rs_to_double_kernel<<<grid, 256, 0, st>>>(src, cur, (int64_t)in_shape[0] * in_shape[1] * in_shape[2]);
    coef = cur;
  }
  RsParams p;
  for (int a = 0; a < 3; ++a) {
    RsAxis& x = p.ax[a];
    x.n_in = in_shape[a]; x.n_out = out_shape[a];
    x.mode = a == separate_axis ? 0 : order;
    x.margin = (order == 3 && a != separate_axis) ? RS_MARGIN : 0;
    x.scale = (double)in_shape[a] / (double)out_shape[a];
  }
  p.clip_axis = separate_axis;
  p.out_mode = out_mode;
  if (order == 0) p.clip_axis = -1;
  rs_gather_kernel<<<grid, 256, 0, st>>>(coef, dst, p, range);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int dwmh_cascade_onehot(int32_t device, const uint8_t* labels, const int32_t in_shape[3], float* dst, const int32_t out_shape[3],
                                   int32_t num_classes, void* stream_) {
  if (!labels || !dst || !in_shape || !out_shape) return fail("dwmh_cascade_onehot: null argument");
  if (num_classes < 2 || num_classes > DWMH_MAX_CLASSES)
    return fail("dwmh_cascade_onehot: num_classes=%d unsupported (2 <= num_classes <= %d)", num_classes, DWMH_MAX_CLASSES);
  for (int a = 0; a < 3; ++a)
    if (in_shape[a] <= 0 || out_shape[a] <= 0)
      return fail("dwmh_cascade_onehot: empty extent on axis %d (in %d, out %d)", a, in_shape[a], out_shape[a]);
  DEV_GUARD(device);
  RsParams p;
  for (int a = 0; a < 3; ++a) {
    RsAxis& x = p.ax[a];
    x.n_in = in_shape[a]; x.n_out = out_shape[a];
    x.mode = 1; x.margin = 0;
    x.scale = (double)in_shape[a] / (double)out_shape[a];
  }
  p.clip_axis = -1;
  p.out_mode = 0;
  rs_onehot_kernel<<<sm_count(device) * 8, 256, 0, (cudaStream_t)stream_>>>(labels, dst, p, num_classes);
  CU_TRY(cudaGetLastError());
  return 0;
}
