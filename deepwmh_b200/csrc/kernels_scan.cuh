// HBM-bound kernels of the path: masked z-score, fused norm+head+softmax, mirror/Gaussian
// overlap-add aggregation, finalize (divide + argmax), small vector helpers.
// Reference semantics: SURVEY.md section 8a rows a2, a11, a12 (nnU-Net v1, un-vendored).
#pragma once
#include "common.cuh"

namespace dwmh {

// ---------------------------------------------------------------------------------------------
// a2  z-score: x = (x - mean) / (std + 1e-8) over the mask, population std, statistics in fp64 (12 B/voxel algorithmic:
// read, read, write).  128-bit coalesced accesses, grid = multiple of the SM count.
// mask_mode 0: all voxels; 1: seg[i] >= 0; 2: vol[i] != 0.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void zscore_stats(const double* acc, float& mean, float& denom) {
  const double cnt = acc[2] > 0.0 ? acc[2] : 1.0;
  const double m = acc[0] / cnt;
  double var = acc[1] / cnt - m * m;
  var = var > 0.0 ? var : 0.0;
  mean = (float)m;
  denom = (float)sqrt(var) + 1e-8f;     // fp32 add, as numpy does with a float32 scalar
}

// One cooperative launch for the whole z-score (volumes of DeepWMH's size are launch-latency bound: 29 MB is 4 us of
// HBM time).  Every CTA reduces its share in fp64 and leaves {sum, sum of squares, count} in its own slot; a grid-wide
// barrier (all CTAs are co-resident: cudaLaunchCooperativeKernel); every CTA then adds the slots in index order --
// deterministic, no atomics on the data, no memset -- and applies the normalisation to the share it already read (the
// second read is served by L2 for volumes below its 126 MB).  slots: [gridDim.x][3] doubles; barrier: one monotonically
// increasing counter, `target` = its value once every CTA of THIS launch has arrived; out_stats (may be null) = the
// totals for the host.
__global__ void __launch_bounds__(256) zscore_fused_kernel(float* __restrict__ vol, const int8_t* __restrict__ seg, int64_t n, int mask_mode,
                                                           double* __restrict__ slots, unsigned long long* __restrict__ barrier,
                                                           unsigned long long target, double* __restrict__ out_stats) {
  double s = 0.0, ss = 0.0, cnt = 0.0;
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  float4* v4 = reinterpret_cast<float4*>(vol);
  const char4* s4 = reinterpret_cast<const char4*>(seg);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = v4[i];
    bool m0 = true, m1 = true, m2 = true, m3 = true;
    if (mask_mode == 1) { const char4 g = s4[i]; m0 = g.x >= 0; m1 = g.y >= 0; m2 = g.z >= 0; m3 = g.w >= 0; }
    else if (mask_mode == 2) { m0 = v.x != 0.f; m1 = v.y != 0.f; m2 = v.z != 0.f; m3 = v.w != 0.f; }
    const float a = m0 ? v.x : 0.f, b = m1 ? v.y : 0.f, c = m2 ? v.z : 0.f, d = m3 ? v.w : 0.f;
    s += (double)a + (double)b + (double)c + (double)d;
    ss += (double)a * a + (double)b * b + (double)c * c + (double)d * d;
    cnt += (double)((int)m0 + (int)m1 + (int)m2 + (int)m3);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {          // tail (n % 4)
    for (int64_t i = n4 << 2; i < n; ++i) {
      const float v = vol[i];
      const bool m = mask_mode == 0 ? true : (mask_mode == 1 ? seg[i] >= 0 : v != 0.f);
      if (m) { s += v; ss += (double)v * v; cnt += 1.0; }
    }
  }
  s = warp_sum_d(s); ss = warp_sum_d(ss); cnt = warp_sum_d(cnt);
  __shared__ double sh[3][8];
  __shared__ double tot[3];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = s; sh[1][w] = ss; sh[2][w] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < 8; ++k) { sh[0][0] += sh[0][k]; sh[1][0] += sh[1][k]; sh[2][0] += sh[2][k]; }
    double* my = slots + (size_t)blockIdx.x * 3;
    my[0] = sh[0][0]; my[1] = sh[1][0]; my[2] = sh[2][0];
    __threadfence();
    atomicAdd(barrier, 1ull);
    while (*reinterpret_cast<volatile unsigned long long*>(barrier) < target) { }
    __threadfence();
  }
  __syncthreads();
  if (w == 0) {      // ordered total: lane l adds slots l, l + 32, ...; the 32 lane sums are combined in lane order
    double a = 0.0, b = 0.0, c = 0.0;
    const volatile double* vs = slots;
    for (int k = l; k < (int)gridDim.x; k += 32) { a += vs[3 * k]; b += vs[3 * k + 1]; c += vs[3 * k + 2]; }
    for (int k = 0; k < 32; ++k) {
      const double ak = __shfl_sync(0xffffffffu, a, k), bk = __shfl_sync(0xffffffffu, b, k), ck = __shfl_sync(0xffffffffu, c, k);
      if (l == 0) { if (k == 0) { tot[0] = ak; tot[1] = bk; tot[2] = ck; } else { tot[0] += ak; tot[1] += bk; tot[2] += ck; } }
    }
  }
  __syncthreads();
  if (out_stats && blockIdx.x == 0 && threadIdx.x < 3) out_stats[threadIdx.x] = tot[threadIdx.x];
  float mean, denom;
  zscore_stats(tot, mean, denom);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = v4[i];
    bool m0 = true, m1 = true, m2 = true, m3 = true;
    if (mask_mode == 1) { const char4 g = s4[i]; m0 = g.x >= 0; m1 = g.y >= 0; m2 = g.z >= 0; m3 = g.w >= 0; }
    else if (mask_mode == 2) { m0 = v.x != 0.f; m1 = v.y != 0.f; m2 = v.z != 0.f; m3 = v.w != 0.f; }
    v.x = m0 ? (v.x - mean) / denom : 0.f;
    v.y = m1 ? (v.y - mean) / denom : 0.f;
    v.z = m2 ? (v.z - mean) / denom : 0.f;
    v.w = m3 ? (v.w - mean) / denom : 0.f;
    v4[i] = v;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    for (int64_t i = n4 << 2; i < n; ++i) {
      const float v = vol[i];
      const bool m = mask_mode == 0 ? true : (mask_mode == 1 ? seg[i] >= 0 : v != 0.f);
      vol[i] = m ? (v - mean) / denom : 0.f;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Head: InstanceNorm+LeakyReLU of the last decoder conv applied on load, 1x1x1 conv to NC = 2..8 logits
// (seg_outputs[-1], no bias), softmax over classes (inference_apply_nonlin): l_k = sum_c w[k][c] x_c,
// p_k = exp(l_k - max) / sum_k' exp(l_k' - max) in fp32, summed in class order.  One thread per voxel (two when
// C == 32 and V is even), grid.y = sample.  y: [n][C/8][V][8] raw conv output; probs: [n][NC][V] fp32.
// ---------------------------------------------------------------------------------------------
template <int NC>
__device__ __forceinline__ void softmax_nc(const float (&l)[NC], float (&p)[NC]) {
  float m = l[0];
#pragma unroll
  for (int k = 1; k < NC; ++k) m = fmaxf(m, l[k]);
  float e[NC], s = 0.f;
#pragma unroll
  for (int k = 0; k < NC; ++k) { e[k] = expf(l[k] - m); s += e[k]; }
#pragma unroll
  for (int k = 0; k < NC; ++k) p[k] = e[k] / s;
}

template <typename T, int NC>
__global__ void __launch_bounds__(256) head_softmax_kernel(const T* __restrict__ y, NormParams np,
                                                           const float* __restrict__ w_head,   // [NC][C]
                                                           float* __restrict__ probs, int C, int64_t V) {
  extern __shared__ __align__(16) float sm[];          // a[C], b[C], w[NC][C]
  float* sa = sm; float* sb = sm + C; float* sw = sm + 2 * C;
  const int n = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 1.f, b = 0.f;
    if (np.sums) norm_coeffs(np, n, C, c, a, b);
    sa[c] = a; sb[c] = b;
  }
  for (int i = threadIdx.x; i < NC * C; i += blockDim.x) sw[i] = w_head[i];
  __syncthreads();
  if (C == 32 && (V & 1) == 0) {
    // the usual head, two voxels per thread (grid sized for V / 2): four 256-bit loads in flight, coefficients read from shared
    // memory as float4 and used for both voxels -- one voxel per thread with scalar coefficient reads was bound by instruction
    // issue (~330 instructions per voxel, 4.9 TB/s), not by HBM.  Same arithmetic order per voxel.
    const int64_t v2 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (2 * v2 >= V) return;
    const uint4* yp2 = reinterpret_cast<const uint4*>(y) + (size_t)n * 4 * V + 2 * v2;
    uint4 q[4][2];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) ld_global_256(yp2 + (size_t)cc * V, q[cc][0], q[cc][1]);
    float l[2][NC];
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
      for (int k = 0; k < NC; ++k) l[e][k] = 0.f;
    const float4* sa4 = reinterpret_cast<const float4*>(sa); const float4* sb4 = reinterpret_cast<const float4*>(sb);
    const float4* sw4 = reinterpret_cast<const float4*>(sw);
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      float f[2][8];
      unpack8<T>(q[cc][0], f[0]); unpack8<T>(q[cc][1], f[1]);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 a4 = sa4[cc * 2 + h], b4 = sb4[cc * 2 + h];
        const float ca[4] = {a4.x, a4.y, a4.z, a4.w}, cb[4] = {b4.x, b4.y, b4.z, b4.w};
        float x[2][4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) x[e][j] = np.sums ? lrelu(fmaf(ca[j], f[e][h * 4 + j], cb[j])) : f[e][h * 4 + j];
#pragma unroll
        for (int k = 0; k < NC; ++k) {
          const float4 u4 = sw4[k * 8 + cc * 2 + h];
          const float cu[4] = {u4.x, u4.y, u4.z, u4.w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) l[e][k] = fmaf(cu[j], x[e][j], l[e][k]);
        }
      }
    }
    float p[2][NC];
    softmax_nc<NC>(l[0], p[0]);
    softmax_nc<NC>(l[1], p[1]);
#pragma unroll
    for (int k = 0; k < NC; ++k)
      *reinterpret_cast<float2*>(probs + ((size_t)n * NC + k) * V + 2 * v2) = make_float2(p[0][k], p[1][k]);
    return;
  }
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const uint4* yp = reinterpret_cast<const uint4*>(y) + (size_t)n * (C >> 3) * V + v;
  float l[NC];
#pragma unroll
  for (int k = 0; k < NC; ++k) l[k] = 0.f;
  auto add_chunk = [&](const uint4& q, int cc) {
    float f[8];
    unpack8<T>(q, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = cc * 8 + j;
      const float x = np.sums ? lrelu(fmaf(sa[c], f[j], sb[c])) : f[j];
#pragma unroll
      for (int k = 0; k < NC; ++k) l[k] = fmaf(sw[k * C + c], x, l[k]);
    }
  };
  if (C == 32) {          // all four channel chunks in flight before the first use
    uint4 q[4];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) q[cc] = ld_stream(yp + (size_t)cc * V);
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) add_chunk(q[cc], cc);
  } else {
    for (int cc = 0; cc < (C >> 3); ++cc) add_chunk(ld_stream(yp + (size_t)cc * V), cc);
  }
  float p[NC];
  softmax_nc<NC>(l, p);
#pragma unroll
  for (int k = 0; k < NC; ++k) probs[((size_t)n * NC + k) * V + v] = p[k];
}

// ---------------------------------------------------------------------------------------------
// a11/a12  One tile: result = sum_m (1/M) * unflip_m(p_m); result *= gaussian; agg[:, tile] += result;
// wgt[tile] += gaussian.  Same fp32 operation order as the reference, per class.  Tiles are aggregated by
// consecutive launches on one stream, so the overlap-add is deterministic (no atomics).
// probs: [M][NC][P] for this tile; metas[m].flip gives the mirror of sample m.
// ---------------------------------------------------------------------------------------------
template <int NC>
__global__ void __launch_bounds__(256) aggregate_tile_kernel(const float* __restrict__ probs,
                                                             const SampleMeta* __restrict__ metas, int M,
                                                             const float* __restrict__ gauss,   // [P] or nullptr
                                                             float* __restrict__ agg, float* __restrict__ wgt,
                                                             int px, int py, int pz, int X, int Y, int Z) {
  const int64_t P = (int64_t)px * py * pz;
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= P) return;
  const int k = (int)(v % pz);
  const int j = (int)((v / pz) % py);
  const int i = (int)(v / ((int64_t)pz * py));
  const float inv = 1.0f / (float)M;
  float r[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) r[c] = 0.f;
  for (int m = 0; m < M; ++m) {
    const int f = metas[m].flip;
    const int kk = (f & 1) ? pz - 1 - k : k;
    const int jj = (f & 2) ? py - 1 - j : j;
    const int ii = (f & 4) ? px - 1 - i : i;
    const int64_t src = ((int64_t)ii * py + jj) * pz + kk;
#pragma unroll
    for (int c = 0; c < NC; ++c) r[c] += inv * probs[((size_t)m * NC + c) * P + src];
  }
  const float g = gauss ? gauss[v] : 1.0f;
  const int64_t V = (int64_t)X * Y * Z;
  const int64_t dst = ((int64_t)(metas[0].ox + i) * Y + (metas[0].oy + j)) * Z + (metas[0].oz + k);
  // agg += r * g.  Two classes round the product before the add (the reference's `*=` then `+=`); more classes add it with
  // one rounding, as the separate kernel these counts ran on was compiled to.  The intrinsics pin both, so every class count
  // keeps its earlier results.  With g = 1 (no Gaussian) both are the plain sum.
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    float& a = agg[(size_t)c * V + dst];
    if constexpr (NC == 2) a = __fadd_rn(a, __fmul_rn(r[c], g));
    else a = __fmaf_rn(r[c], g, a);
  }
  wgt[dst] += g;
}

// ---------------------------------------------------------------------------------------------
// a12, tile-sharded mode: the weight buffer is data-independent, so a rank computes ALL of it locally instead of
// reducing it over NVLink.  Per voxel the importance map of every covering tile is added in tile order (x outer, z
// inner) -- the fp32 sequence the per-tile overlap-add of a single-GPU run performs, hence bit-identical to it.
// ---------------------------------------------------------------------------------------------
constexpr int WM_MAX_STEPS = 64;
struct TileSteps { int n[3]; int s[3][WM_MAX_STEPS]; };

__global__ void __launch_bounds__(256) weight_map_kernel(const float* __restrict__ gauss, float* __restrict__ wgt, TileSteps ts,
                                                         int px, int py, int pz, int X, int Y, int Z) {
  const int64_t V = (int64_t)X * Y * Z;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += stride) {
    const int z = (int)(v % Z), y = (int)((v / Z) % Y), x = (int)(v / ((int64_t)Z * Y));
    float w = 0.f;
    for (int ix = 0; ix < ts.n[0]; ++ix) {
      const int i = x - ts.s[0][ix];
      if ((unsigned)i >= (unsigned)px) continue;
      for (int iy = 0; iy < ts.n[1]; ++iy) {
        const int j = y - ts.s[1][iy];
        if ((unsigned)j >= (unsigned)py) continue;
        for (int iz = 0; iz < ts.n[2]; ++iz) {
          const int k = z - ts.s[2][iz];
          if ((unsigned)k >= (unsigned)pz) continue;
          w += gauss ? __ldg(gauss + ((int64_t)i * py + j) * pz + k) : 1.0f;
        }
      }
    }
    wgt[v] = w;
  }
}

// ---------------------------------------------------------------------------------------------
// a12 tail: class_probabilities = agg / wgt; seg = argmax (first maximum, numpy.argmax).  (8 NC + 5) B/voxel.
// ---------------------------------------------------------------------------------------------
// p[c] /= w for every class; returns the first class holding the maximum
template <int NC>
__device__ __forceinline__ uint8_t divide_argmax(float (&p)[NC], float w) {
  p[0] = p[0] / w;
  float best = p[0];
  int arg = 0;
#pragma unroll
  for (int c = 1; c < NC; ++c) {
    p[c] = p[c] / w;
    if (p[c] > best) { best = p[c]; arg = c; }
  }
  return (uint8_t)arg;
}

// softmax_out [NC][V] may alias agg (in-place normalisation): neither is __restrict__, and every thread reads all of its
// elements before it writes them.
template <int NC, bool VEC>      // VEC: V % 4 == 0 and every buffer 16-byte (seg: 4-byte) aligned
__global__ void __launch_bounds__(256) finalize_kernel(const float* agg, const float* __restrict__ wgt,
                                                       float* softmax_out, uint8_t* __restrict__ seg, int64_t V) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if constexpr (VEC) {
    // 128-bit accesses (four voxels per thread and step): the pass is a pure stream, bound by bytes in flight.  The class
    // planes are reached by stepping one pointer (a pointer per class, hoisted out of the loop, made ptxas spill at NC = 7).
    const int64_t V4 = V >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < V4; i += stride) {
      const float4 w = reinterpret_cast<const float4*>(wgt)[i];
      float p[4][NC];
      const float4* a = reinterpret_cast<const float4*>(agg) + i;
#pragma unroll
      for (int c = 0; c < NC; ++c, a += V4) {
        const float4 x = *a;
        p[0][c] = x.x; p[1][c] = x.y; p[2][c] = x.z; p[3][c] = x.w;
      }
      const uchar4 s = make_uchar4(divide_argmax<NC>(p[0], w.x), divide_argmax<NC>(p[1], w.y), divide_argmax<NC>(p[2], w.z),
                                   divide_argmax<NC>(p[3], w.w));
      if (softmax_out) {
        float4* o = reinterpret_cast<float4*>(softmax_out) + i;
#pragma unroll
        for (int c = 0; c < NC; ++c, o += V4) *o = make_float4(p[0][c], p[1][c], p[2][c], p[3][c]);
      }
      if (seg) reinterpret_cast<uchar4*>(seg)[i] = s;
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += stride) {
      float p[NC];
#pragma unroll
      for (int c = 0; c < NC; ++c) p[c] = agg[(size_t)c * V + i];
      const uint8_t s = divide_argmax<NC>(p, wgt[i]);
      if (softmax_out) {
#pragma unroll
        for (int c = 0; c < NC; ++c) softmax_out[(size_t)c * V + i] = p[c];
      }
      if (seg) seg[i] = s;
    }
  }
}

// argmax over NC classes of p [NC][V], first maximum (numpy.argmax)
__global__ void __launch_bounds__(256) argmax_kernel(const float* __restrict__ p, int NC, uint8_t* __restrict__ seg, int64_t V) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += stride) {
    float best = p[i];
    int arg = 0;
    for (int c = 1; c < NC; ++c) {
      const float x = p[(size_t)c * V + i];
      if (x > best) { best = x; arg = c; }
    }
    seg[i] = (uint8_t)arg;
  }
}

__global__ void __launch_bounds__(256) axpy_kernel(float* __restrict__ acc, const float* __restrict__ x, float alpha, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) acc[i] = fmaf(alpha, x[i], acc[i]);
}

// SURVEY 8f-3: checkpoint ensemble of masked background probabilities (deepwmh/pipeline/DCNN_multistage.py:102-125).
//   y = 1 - m (1 - x)            per checkpoint, float32 arrays (load_nifti_simple), one rounding per operation (:108-109)
//   field += y                    float32 running field (:115-117)
// and after the k checkpoints: field /= k; label = field < 0.5 (:118-119).
__global__ void __launch_bounds__(256) ensemble_masked_add_kernel(float* __restrict__ acc, const float* __restrict__ x,
                                                                  const float* __restrict__ m, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    // float32 arithmetic, one rounding per operation, as numpy evaluates 1-(m*(1-x)) on the float32 arrays that
    // load_nifti_simple returns (deepwmh/utilities/data_io.py:288-290); no FMA contraction
    const float mv = m ? m[i] : 1.f;
    const float y = __fsub_rn(1.f, __fmul_rn(mv, __fsub_rn(1.f, x[i])));
    acc[i] = __fadd_rn(acc[i], y);
  }
}
__global__ void __launch_bounds__(256) ensemble_refine_kernel(float* __restrict__ acc, float k, uint8_t* __restrict__ label, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float f = acc[i] / k;
    acc[i] = f;
    if (label) label[i] = f < 0.5f ? 1 : 0;
  }
}

// chunked T [n][C/8][V][8] -> fp32 NCDHW (debug / layer-level parity tests), optional norm+lrelu
template <typename T>
__global__ void __launch_bounds__(256) unpack_layer_kernel(const T* __restrict__ y, NormParams np, float* __restrict__ out,
                                                           int N, int C, int64_t V) {
  const int64_t total = (int64_t)N * (C >> 3) * V;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t v = i % V;
    const int cc = (int)((i / V) % (C >> 3));
    const int n = (int)(i / (V * (C >> 3)));
    float f[8];
    unpack8<T>(reinterpret_cast<const uint4*>(y)[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float x = f[j];
      if (np.sums) { float a, b; norm_coeffs(np, n, C, cc * 8 + j, a, b); x = lrelu(fmaf(a, x, b)); }
      out[((size_t)n * C + cc * 8 + j) * V + v] = x;
    }
  }
}

}  // namespace dwmh
