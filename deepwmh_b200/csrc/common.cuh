// Shared device helpers: activation storage type traits, chunked layout indexing, reductions.
//
// Activation layout in HBM ("NC8": channel chunks of 8, 16 bytes per voxel-chunk):
//   act[n][c/8][d][h][w][c%8]   element type T = __half (default) or __nv_bfloat16
// d/h/w are the x/y/z axes of nnU-Net's (c, x, y, z) arrays (z fastest).  One 16-byte vector holds
// 8 channels of one voxel; this is the tcgen05 "K-major, no swizzle" core-matrix row, so a TMA box
// of a [c/8][h][w] slab lands in shared memory directly as a valid UMMA operand.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace dwmh {

template <typename T> struct ActT;
template <> struct ActT<__half> {
  using T2 = __half2;
  static __device__ __forceinline__ float2 to_f2(uint32_t u) { return __half22float2(*reinterpret_cast<__half2*>(&u)); }
  static __device__ __forceinline__ uint32_t from_f2(float a, float b) { __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }
  static __device__ __forceinline__ float to_f(__half h) { return __half2float(h); }
  static __device__ __forceinline__ __half from_f(float f) { return __float2half_rn(f); }
  static constexpr int kUmmaFormat = 0;   // F16
};
template <> struct ActT<__nv_bfloat16> {
  using T2 = __nv_bfloat162;
  static __device__ __forceinline__ float2 to_f2(uint32_t u) { return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u)); }
  static __device__ __forceinline__ uint32_t from_f2(float a, float b) { __nv_bfloat162 h = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }
  static __device__ __forceinline__ float to_f(__nv_bfloat16 h) { return __bfloat162float(h); }
  static __device__ __forceinline__ __nv_bfloat16 from_f(float f) { return __float2bfloat16_rn(f); }
  static constexpr int kUmmaFormat = 1;   // BF16
};

// 8 channels of one voxel <-> 8 floats
template <typename T>
__device__ __forceinline__ void unpack8(const uint4& v, float f[8]) {
  float2 a = ActT<T>::to_f2(v.x), b = ActT<T>::to_f2(v.y), c = ActT<T>::to_f2(v.z), d = ActT<T>::to_f2(v.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
template <typename T>
__device__ __forceinline__ uint4 pack8(const float f[8]) {
  uint4 v;
  v.x = ActT<T>::from_f2(f[0], f[1]); v.y = ActT<T>::from_f2(f[2], f[3]);
  v.z = ActT<T>::from_f2(f[4], f[5]); v.w = ActT<T>::from_f2(f[6], f[7]);
  return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Ordered grid reduction of the cooperative statistics kernels (256 threads, every CTA resident) over each thread's
// (s, ss, cnt).  Every CTA leaves its {sum, sum of squares, count} in its slot (slots: [gridDim.x][3] doubles), arrives at
// `barrier` and waits until the counter reaches `target`; warp 0 then adds the slots in index order -- deterministic, no
// atomics on the data, the same totals in every CTA.  Returns the totals, in shared memory; out_stats (may be null)
// receives them from CTA 0.
__device__ __forceinline__ const double* grid_ordered_totals(double s, double ss, double cnt, double* __restrict__ slots,
                                                             unsigned long long* __restrict__ barrier, unsigned long long target,
                                                             double* __restrict__ out_stats) {
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
  return tot;
}

// order-preserving float <-> unsigned key (atomicMin / atomicMax on floats)
__device__ __forceinline__ unsigned float_key(float f) { const unsigned u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float key_float(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

__device__ __forceinline__ float lrelu(float v) { return v > 0.f ? v : 0.01f * v; }

// streaming 128-bit accesses that do not pollute L1
__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

__device__ __forceinline__ void st_shared_128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// 256-bit global accesses (sm_100): two 16-byte voxel-chunks per instruction keep twice the bytes in flight per thread;
// the pass is a pure stream and was bound by memory-level parallelism (2048 threads x 16 B per SM).
__device__ __forceinline__ void ld_global_256(const void* p, uint4& a, uint4& b) {
  asm volatile("ld.global.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}
__device__ __forceinline__ void st_global_256(void* p, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}

// Per-forward sample descriptor: where the patch sits in the padded volume and which axes are mirrored.
struct SampleMeta {
  int32_t ox, oy, oz;     // tile origin in the volume (axis 0,1,2)
  int32_t flip;           // bit0: flip axis 2 (z), bit1: axis 1 (y), bit2: axis 0 (x)   == mirror index m
};

// InstanceNorm statistics of one layer, fp64, two formats:
//   inv_count  > 0: sums[(n*C + c)*2 + {0,1}] = {sum y, sum y^2}          (CUDA-core cross-check kernels: fp64 atomics)
//   inv_count == 0: sums[(n*C + c)*2 + {0,1}] = {mean, biased variance}    (tcgen05 path: written by stats_reduce_kernel from
//                   the per-CTA Welford partials in a fixed order -- deterministic and free of E[x^2] - E[x]^2 cancellation)
struct NormParams {
  const double* sums;     // nullptr => identity (no norm / activation)
  const float* gamma;
  const float* beta;
  double inv_count;       // 1 / (D*H*W), or 0 (see above)
};

// a = gamma / sqrt(var + eps), b = beta - mean * a   (InstanceNorm3d eps 1e-5, biased variance)
__device__ __forceinline__ void norm_coeffs(const NormParams& np, int n, int C, int c, float& a, float& b) {
  const double s1 = np.sums[((size_t)n * C + c) * 2 + 0];
  const double s2 = np.sums[((size_t)n * C + c) * 2 + 1];
  double mean = s1, var = s2;
  if (np.inv_count != 0.0) {
    mean = s1 * np.inv_count;
    var = s2 * np.inv_count - mean * mean;
  }
  var = var > 0.0 ? var : 0.0;
  const double inv = rsqrt(var + 1e-5);
  a = (float)((double)np.gamma[c] * inv);
  b = (float)((double)np.beta[c] - mean * (double)np.gamma[c] * inv);
}

// One (count, mean, M2 = sum (x - mean)^2) partial of the tcgen05 conv epilogue: one per (work item, channel).
struct StatPartial { float n, mean, m2, pad; };

// Chan's pairwise update of (n, mean, M2) with a second partial; exact in real arithmetic, well conditioned in floating point.
template <typename F>
__device__ __forceinline__ void stat_merge(F& n, F& mean, F& m2, F nb, F meanb, F m2b) {
  const F nt = n + nb;
  const F w = nt > (F)0 ? nb / nt : (F)0;
  const F d = meanb - mean;
  mean = mean + d * w;
  m2 = m2 + m2b + d * d * n * w;
  n = nt;
}

}  // namespace dwmh
