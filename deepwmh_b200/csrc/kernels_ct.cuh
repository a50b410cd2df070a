// nnU-Net's CT intensity normalisation schemes [U:GenericPreprocessor.resample_and_normalize], per modality after the
// spacing resample, in fp32 with the plans' constants rounded to fp32 (upstream applies python floats to float32 arrays,
// which numpy 1.x evaluates in float32):
//   "CT":  x = (clip(x, lb, ub) - mean) / sd                                          (mean, sd from the plans)
//   "CT2": mask = lb < x < ub (unclipped); x = clip(x, lb, ub); x = (x - mn) / sd      (mn, sd of x over mask, population sd)
// then, for a modality with use_mask_for_norm, x = 0 where the crop mask seg < 0.  IEEE division, no reciprocal.
// clip keeps a NaN (numpy.clip does); both passes are pure HBM streams (8 B/voxel, + 1 B with seg).
#pragma once
#include "common.cuh"

namespace dwmh {

__device__ __forceinline__ float ct_clip(float x, float lb, float ub) { return x < lb ? lb : (x > ub ? ub : x); }

// `/` is the IEEE division under nvcc's default -prec-div=true (the __fdiv_rn intrinsic made ptxas spill in ct2_fused_kernel)
__device__ __forceinline__ float ct_apply(float x, float lb, float ub, float mean, float sd) {
  return (ct_clip(x, lb, ub) - mean) / sd;
}

// "CT" with the plans' constants.  VEC: vol 16-byte and seg 4-byte aligned -- four voxels per thread and step with 128-bit
// loads and stores, the n % 4 tail by scalar accesses; otherwise every voxel is a scalar access.  seg may be null (no
// zeroing).
template <bool VEC>
__global__ void __launch_bounds__(256) ct_normalize_kernel(float* __restrict__ vol, const int8_t* __restrict__ seg, int64_t n,
                                                           float lb, float ub, float mean, float sd) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t done = 0;
  if constexpr (VEC) {
    const int64_t n4 = n >> 2;
    float4* v4 = reinterpret_cast<float4*>(vol);
    const char4* s4 = reinterpret_cast<const char4*>(seg);
    for (int64_t i = t; i < n4; i += stride) {
      float4 v = ld_stream_f4(v4 + i);
      v.x = ct_apply(v.x, lb, ub, mean, sd); v.y = ct_apply(v.y, lb, ub, mean, sd);
      v.z = ct_apply(v.z, lb, ub, mean, sd); v.w = ct_apply(v.w, lb, ub, mean, sd);
      if (seg) {
        const char4 g = s4[i];
        if (g.x < 0) v.x = 0.f;
        if (g.y < 0) v.y = 0.f;
        if (g.z < 0) v.z = 0.f;
        if (g.w < 0) v.w = 0.f;
      }
      v4[i] = v;
    }
    done = n4 << 2;
  }
  for (int64_t i = done + t; i < n; i += stride) {
    const float x = ct_apply(vol[i], lb, ub, mean, sd);
    vol[i] = (seg && seg[i] < 0) ? 0.f : x;
  }
}

// CT2's statistics of one voxel: inside (lb, ub), which clip leaves as it is
__device__ __forceinline__ void ct2_add(float x, float lb, float ub, double& s, double& ss, double& cnt) {
  if (x > lb && x < ub) { s += x; ss += (double)x * x; cnt += 1.0; }
}

// "CT2": one cooperative launch, as zscore_fused_kernel: every thread sums its voxels inside (lb, ub) in fp64, the CTAs
// leave {sum, sum of squares, count} in their slots, a grid-wide barrier, every CTA adds the slots in index order
// (grid_ordered_totals: deterministic, no atomics on the data) and normalises the share it read.  vol 16-byte, seg 4-byte
// aligned.  slots: [gridDim.x][3] doubles; barrier: a counter that is `target` once every CTA of this launch has arrived;
// out_stats (may be null) = the totals.  An empty mask gives NaN (0 / 0), as upstream; the caller refuses it from the count.
__global__ void __launch_bounds__(256) ct2_fused_kernel(float* __restrict__ vol, const int8_t* __restrict__ seg, int64_t n,
                                                        float lb, float ub, double* __restrict__ slots,
                                                        unsigned long long* __restrict__ barrier, unsigned long long target,
                                                        double* __restrict__ out_stats) {
  double s = 0.0, ss = 0.0, cnt = 0.0;
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  float4* v4 = reinterpret_cast<float4*>(vol);
  const char4* s4 = reinterpret_cast<const char4*>(seg);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = v4[i];
    ct2_add(v.x, lb, ub, s, ss, cnt); ct2_add(v.y, lb, ub, s, ss, cnt);
    ct2_add(v.z, lb, ub, s, ss, cnt); ct2_add(v.w, lb, ub, s, ss, cnt);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (int64_t i = n4 << 2; i < n; ++i) ct2_add(vol[i], lb, ub, s, ss, cnt);
  const double* tot = grid_ordered_totals(s, ss, cnt, slots, barrier, target, out_stats);
  const double m = tot[0] / tot[2];
  double var = tot[1] / tot[2] - m * m;
  var = var > 0.0 ? var : 0.0;
  const float mean = (float)m, sd = (float)sqrt(var);        // numpy's float32 mean() / std() are float32 scalars
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = v4[i];
    v.x = ct_apply(v.x, lb, ub, mean, sd); v.y = ct_apply(v.y, lb, ub, mean, sd);
    v.z = ct_apply(v.z, lb, ub, mean, sd); v.w = ct_apply(v.w, lb, ub, mean, sd);
    if (seg) {
      const char4 g = s4[i];
      if (g.x < 0) v.x = 0.f;
      if (g.y < 0) v.y = 0.f;
      if (g.z < 0) v.z = 0.f;
      if (g.w < 0) v.w = 0.f;
    }
    v4[i] = v;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    for (int64_t i = n4 << 2; i < n; ++i) {
      const float x = ct_apply(vol[i], lb, ub, mean, sd);
      vol[i] = (seg && seg[i] < 0) ? 0.f : x;
    }
  }
}

}  // namespace dwmh
