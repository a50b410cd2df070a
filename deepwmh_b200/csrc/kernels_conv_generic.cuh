// CUDA-core kernels that cover every layer shape of Generic_UNet (any kernel in {1,3}^3, stride in
// {1,2}^3, k=s transposed conv).  They are the shape-complete implementation; the tcgen05 implicit
// GEMM (conv_tcgen05.cuh) takes over the layer shapes it supports and is cross-checked against these.
// fp32 accumulate; raw outputs stored as T with per-(sample, channel) sum / sum-of-squares in fp64 for
// InstanceNorm.  Conv bias is not applied: it cancels exactly under InstanceNorm.
// Reference semantics: Generic_UNet.forward / ConvDropoutNormNonlin [U:generic_UNet.py], SURVEY.md A1.
#pragma once
#include "common.cuh"

namespace dwmh {
__host__ __device__ inline int tc_s2d_class(int d, int h, int w, int sd, int sh, int sw);


// ---------------------------------------------------------------------------------------------
// First conv (Cin == 1) fused with tile extraction + mirror flip: reads the normalised fp32 volume
// (or fp32 patches) directly, writes raw [n][Cout/8][P][8] + statistics.  One thread per output
// voxel, 8 output channels at a time.  w: [taps][Cout] fp32.
// ---------------------------------------------------------------------------------------------
struct FirstConvParams {
  const float* src;            // volume [SX][SY][SZ] (patch_mode 0) or patches [n][px][py][pz] (1)
  const SampleMeta* metas;     // per sample origin + flip (patch_mode 0)
  const float* w;              // [kd*kh*kw][Cout]
  void* out;
  double* sums;                // [n][Cout][2]
  int patch_mode;
  int SX, SY, SZ;
  int px, py, pz;
  int kd, kh, kw;
  int Cout;
  int Cin;                     // modalities (conv_first_mm_kernel; the single-modality kernels ignore it)
  int64_t mstride;             // floats between two modalities of the volume (patch_mode 0)
};

// K3: kernel is 3x3x3 (fully unrolled taps, inputs stay in registers).  Each thread walks FC_VPT voxels
// (stride = blockDim) and keeps per-channel running statistics in registers (Cout <= 32) so the warp
// reduction happens once per thread instead of once per voxel.
constexpr int FC_VPT = 4;

template <typename T, bool K3>
__global__ void __launch_bounds__(256) conv_first_kernel(FirstConvParams p) {
  extern __shared__ float smf[];                 // weights [taps][Cout], then stats [Cout][2]
  const int kd = K3 ? 3 : p.kd, kh = K3 ? 3 : p.kh, kw = K3 ? 3 : p.kw;
  const int taps = kd * kh * kw;
  float* sw = smf;
  float* sstat = smf + taps * p.Cout;
  for (int i = threadIdx.x; i < taps * p.Cout; i += blockDim.x) sw[i] = p.w[i];
  for (int i = threadIdx.x; i < 2 * p.Cout; i += blockDim.x) sstat[i] = 0.f;
  __syncthreads();
  const int n = blockIdx.y;
  const int64_t P = (int64_t)p.px * p.py * p.pz;
  int ox = 0, oy = 0, oz = 0, flip = 0;
  const float* src = p.src;
  int SY = p.SY, SZ = p.SZ;
  if (p.patch_mode) { src += (size_t)n * P; SY = p.py; SZ = p.pz; }
  else { const SampleMeta m = p.metas[n]; ox = m.ox; oy = m.oy; oz = m.oz; flip = m.flip; }
  const int lane = threadIdx.x & 31;
  const bool reg_stats = p.Cout <= 32;
  float rs[32], rq[32];
#pragma unroll
  for (int q = 0; q < 32; ++q) { rs[q] = 0.f; rq[q] = 0.f; }
  for (int it = 0; it < FC_VPT; ++it) {
    const int64_t v = ((int64_t)blockIdx.x * FC_VPT + it) * blockDim.x + threadIdx.x;
    const bool active = v < P;
    const int k = (int)(v % p.pz), j = (int)((v / p.pz) % p.py), i = (int)(v / ((int64_t)p.pz * p.py));
    float xin[27];
#pragma unroll
    for (int a = 0; a < (K3 ? 3 : 3); ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          float val = 0.f;
          if (a < kd && b < kh && c < kw) {
            const int ii = i + a - (kd >> 1), jj = j + b - (kh >> 1), kk = k + c - (kw >> 1);
            if (active && ii >= 0 && ii < p.px && jj >= 0 && jj < p.py && kk >= 0 && kk < p.pz) {
              const int si = ox + ((flip & 4) ? p.px - 1 - ii : ii);
              const int sj = oy + ((flip & 2) ? p.py - 1 - jj : jj);
              const int sk = oz + ((flip & 1) ? p.pz - 1 - kk : kk);
              val = __ldg(src + ((size_t)si * SY + sj) * SZ + sk);
            }
          }
          xin[(a * 3 + b) * 3 + c] = val;
        }
    uint4* outp = reinterpret_cast<uint4*>(p.out) + (size_t)n * (p.Cout >> 3) * P + v;
    for (int cc = 0; cc < (p.Cout >> 3); ++cc) {
      float acc[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q] = 0.f;
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            if (a < kd && b < kh && c < kw) {
              const int t = (a * kh + b) * kw + c;
              const float4 w0 = *reinterpret_cast<const float4*>(sw + t * p.Cout + cc * 8);
              const float4 w1 = *reinterpret_cast<const float4*>(sw + t * p.Cout + cc * 8 + 4);
              const float x = xin[(a * 3 + b) * 3 + c];
              acc[0] = fmaf(x, w0.x, acc[0]); acc[1] = fmaf(x, w0.y, acc[1]); acc[2] = fmaf(x, w0.z, acc[2]); acc[3] = fmaf(x, w0.w, acc[3]);
              acc[4] = fmaf(x, w1.x, acc[4]); acc[5] = fmaf(x, w1.y, acc[5]); acc[6] = fmaf(x, w1.z, acc[6]); acc[7] = fmaf(x, w1.w, acc[7]);
            }
          }
      if (active) outp[(size_t)cc * P] = pack8<T>(acc);
      if (reg_stats) {
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          if (cc == q4 && active) {
#pragma unroll
            for (int q = 0; q < 8; ++q) { rs[q4 * 8 + q] += acc[q]; rq[q4 * 8 + q] = fmaf(acc[q], acc[q], rq[q4 * 8 + q]); }
          }
        }
      } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float a_ = active ? acc[q] : 0.f;
          const float s = warp_sum(a_), ss = warp_sum(a_ * a_);
          if (lane == 0) { atomicAdd(&sstat[(cc * 8 + q) * 2], s); atomicAdd(&sstat[(cc * 8 + q) * 2 + 1], ss); }
        }
      }
    }
  }
  if (reg_stats) {
    // transposing butterfly: lane l ends with the warp total of channel l
#pragma unroll
    for (int k = 16; k >= 1; k >>= 1) {
      const bool up = (lane & k) != 0;
#pragma unroll
      for (int i = 0; i < k; ++i) {
        const float sa_ = up ? rs[i] : rs[i + k], ka_ = up ? rs[i + k] : rs[i];
        const float sb_ = up ? rq[i] : rq[i + k], kb_ = up ? rq[i + k] : rq[i];
        rs[i] = ka_ + __shfl_xor_sync(0xffffffffu, sa_, k);
        rq[i] = kb_ + __shfl_xor_sync(0xffffffffu, sb_, k);
      }
    }
    if (lane < p.Cout) { atomicAdd(&sstat[lane * 2], rs[0]); atomicAdd(&sstat[lane * 2 + 1], rq[0]); }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * p.Cout; c += blockDim.x)
    atomicAdd(p.sums + (size_t)n * p.Cout * 2 + c, (double)sstat[c]);
}

// 3x3x3 specialisation with TWO z-adjacent voxels per thread: one broadcast weight load feeds 16 FMAs
// (the one-voxel form is bound by the shared-memory port: 1 LDS.128 per 4 FMAs), and the pair shares its
// 3x3x4 input neighbourhood.  Requires pz even and Cout <= 32.
template <typename T>
__global__ void __launch_bounds__(128) conv_first_k3x2_kernel(FirstConvParams p) {
  extern __shared__ float smf[];                 // weights [27][Cout], then stats [Cout][2]
  float* sw = smf;
  float* sstat = smf + 27 * p.Cout;
  for (int i = threadIdx.x; i < 27 * p.Cout; i += blockDim.x) sw[i] = p.w[i];
  for (int i = threadIdx.x; i < 2 * p.Cout; i += blockDim.x) sstat[i] = 0.f;
  __syncthreads();
  const int n = blockIdx.y;
  const int64_t P = (int64_t)p.px * p.py * p.pz, P2 = P >> 1;
  int ox = 0, oy = 0, oz = 0, flip = 0;
  const float* src = p.src;
  int SY = p.SY, SZ = p.SZ;
  if (p.patch_mode) { src += (size_t)n * P; SY = p.py; SZ = p.pz; }
  else { const SampleMeta m = p.metas[n]; ox = m.ox; oy = m.oy; oz = m.oz; flip = m.flip; }
  const int lane = threadIdx.x & 31;
  const int pz2 = p.pz >> 1;
  float rs[32], rq[32];
#pragma unroll
  for (int q = 0; q < 32; ++q) { rs[q] = 0.f; rq[q] = 0.f; }
  for (int it = 0; it < FC_VPT; ++it) {
    const int64_t v2 = ((int64_t)blockIdx.x * FC_VPT + it) * blockDim.x + threadIdx.x;      // voxel-pair index
    const bool active = v2 < P2;
    const int k = (int)(v2 % pz2) * 2, j = (int)((v2 / pz2) % p.py), i = (int)(v2 / ((int64_t)pz2 * p.py));
    float xin[9][4];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int ii = i + a - 1, jj = j + b - 1, kk = k + c - 1;
          float val = 0.f;
          if (active && ii >= 0 && ii < p.px && jj >= 0 && jj < p.py && kk >= 0 && kk < p.pz) {
            const int si = ox + ((flip & 4) ? p.px - 1 - ii : ii);
            const int sj = oy + ((flip & 2) ? p.py - 1 - jj : jj);
            const int sk = oz + ((flip & 1) ? p.pz - 1 - kk : kk);
            val = __ldg(src + ((size_t)si * SY + sj) * SZ + sk);
          }
          xin[a * 3 + b][c] = val;
        }
    const int64_t v = ((int64_t)i * p.py + j) * p.pz + k;
    uint4* outp = reinterpret_cast<uint4*>(p.out) + (size_t)n * (p.Cout >> 3) * P + v;
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      if (cc < (p.Cout >> 3)) {
        float a0[8], a1[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { a0[q] = 0.f; a1[q] = 0.f; }
#pragma unroll
        for (int ab = 0; ab < 9; ++ab)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const float4 w0 = *reinterpret_cast<const float4*>(sw + (ab * 3 + c) * p.Cout + cc * 8);
            const float4 w1 = *reinterpret_cast<const float4*>(sw + (ab * 3 + c) * p.Cout + cc * 8 + 4);
            const float x0 = xin[ab][c], x1 = xin[ab][c + 1];
            a0[0] = fmaf(x0, w0.x, a0[0]); a0[1] = fmaf(x0, w0.y, a0[1]); a0[2] = fmaf(x0, w0.z, a0[2]); a0[3] = fmaf(x0, w0.w, a0[3]);
            a0[4] = fmaf(x0, w1.x, a0[4]); a0[5] = fmaf(x0, w1.y, a0[5]); a0[6] = fmaf(x0, w1.z, a0[6]); a0[7] = fmaf(x0, w1.w, a0[7]);
            a1[0] = fmaf(x1, w0.x, a1[0]); a1[1] = fmaf(x1, w0.y, a1[1]); a1[2] = fmaf(x1, w0.z, a1[2]); a1[3] = fmaf(x1, w0.w, a1[3]);
            a1[4] = fmaf(x1, w1.x, a1[4]); a1[5] = fmaf(x1, w1.y, a1[5]); a1[6] = fmaf(x1, w1.z, a1[6]); a1[7] = fmaf(x1, w1.w, a1[7]);
          }
        if (active) {
          outp[(size_t)cc * P] = pack8<T>(a0);
          outp[(size_t)cc * P + 1] = pack8<T>(a1);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            rs[cc * 8 + q] += a0[q] + a1[q];
            rq[cc * 8 + q] = fmaf(a0[q], a0[q], fmaf(a1[q], a1[q], rq[cc * 8 + q]));
          }
        }
      }
    }
  }
#pragma unroll
  for (int k = 16; k >= 1; k >>= 1) {
    const bool up = (lane & k) != 0;
#pragma unroll
    for (int i = 0; i < k; ++i) {
      const float sa_ = up ? rs[i] : rs[i + k], ka_ = up ? rs[i + k] : rs[i];
      const float sb_ = up ? rq[i] : rq[i + k], kb_ = up ? rq[i + k] : rq[i];
      rs[i] = ka_ + __shfl_xor_sync(0xffffffffu, sa_, k);
      rq[i] = kb_ + __shfl_xor_sync(0xffffffffu, sb_, k);
    }
  }
  if (lane < p.Cout) { atomicAdd(&sstat[lane * 2], rs[0]); atomicAdd(&sstat[lane * 2 + 1], rq[0]); }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * p.Cout; c += blockDim.x)
    atomicAdd(p.sums + (size_t)n * p.Cout * 2 + c, (double)sstat[c]);
}

// ---------------------------------------------------------------------------------------------
// First conv with Cin = p.Cin > 1 modalities (nnU-Net models with several input images): the volume is [Cin][SX][SY][SZ]
// (patch_mode 0, modalities p.mstride floats apart) or patches [n][Cin][px][py][pz].  One thread per output voxel; per
// 8-channel output chunk the taps of modality 0, 1, ... accumulate in that order into one fp32 sum.  w: [Cin][taps][Cout].
// Statistics as in conv_first_kernel.  Requires Cout <= 32.
// ---------------------------------------------------------------------------------------------
template <typename T, bool K3>
__global__ void __launch_bounds__(256) conv_first_mm_kernel(FirstConvParams p) {
  extern __shared__ float smf[];                 // weights [Cin][taps][Cout], then stats [Cout][2]
  const int kd = K3 ? 3 : p.kd, kh = K3 ? 3 : p.kh, kw = K3 ? 3 : p.kw;
  const int taps = kd * kh * kw;
  float* sw = smf;
  float* sstat = smf + p.Cin * taps * p.Cout;
  for (int i = threadIdx.x; i < p.Cin * taps * p.Cout; i += blockDim.x) sw[i] = p.w[i];
  for (int i = threadIdx.x; i < 2 * p.Cout; i += blockDim.x) sstat[i] = 0.f;
  __syncthreads();
  const int n = blockIdx.y;
  const int64_t P = (int64_t)p.px * p.py * p.pz;
  int ox = 0, oy = 0, oz = 0, flip = 0;
  const float* src = p.src;
  int SY = p.SY, SZ = p.SZ;
  int64_t mstride = p.mstride;
  if (p.patch_mode) { src += (size_t)n * p.Cin * P; SY = p.py; SZ = p.pz; mstride = P; }
  else { const SampleMeta m = p.metas[n]; ox = m.ox; oy = m.oy; oz = m.oz; flip = m.flip; }
  const int lane = threadIdx.x & 31;
  float rs[32], rq[32];
#pragma unroll
  for (int q = 0; q < 32; ++q) { rs[q] = 0.f; rq[q] = 0.f; }
  for (int it = 0; it < FC_VPT; ++it) {
    const int64_t v = ((int64_t)blockIdx.x * FC_VPT + it) * blockDim.x + threadIdx.x;
    const bool active = v < P;
    const int k = (int)(v % p.pz), j = (int)((v / p.pz) % p.py), i = (int)(v / ((int64_t)p.pz * p.py));
    float acc[4][8];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc)
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[cc][q] = 0.f;
    for (int m = 0; m < p.Cin; ++m) {
      float xin[27];
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            float val = 0.f;
            if (a < kd && b < kh && c < kw) {
              const int ii = i + a - (kd >> 1), jj = j + b - (kh >> 1), kk = k + c - (kw >> 1);
              if (active && ii >= 0 && ii < p.px && jj >= 0 && jj < p.py && kk >= 0 && kk < p.pz) {
                const int si = ox + ((flip & 4) ? p.px - 1 - ii : ii);
                const int sj = oy + ((flip & 2) ? p.py - 1 - jj : jj);
                const int sk = oz + ((flip & 1) ? p.pz - 1 - kk : kk);
                val = __ldg(src + (size_t)m * mstride + ((size_t)si * SY + sj) * SZ + sk);
              }
            }
            xin[(a * 3 + b) * 3 + c] = val;
          }
      const float* wm = sw + (size_t)m * taps * p.Cout;
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        if (cc < (p.Cout >> 3)) {
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b)
#pragma unroll
              for (int c = 0; c < 3; ++c) {
                if (a < kd && b < kh && c < kw) {
                  const int t = (a * kh + b) * kw + c;
                  const float4 w0 = *reinterpret_cast<const float4*>(wm + t * p.Cout + cc * 8);
                  const float4 w1 = *reinterpret_cast<const float4*>(wm + t * p.Cout + cc * 8 + 4);
                  const float x = xin[(a * 3 + b) * 3 + c];
                  float* ac = acc[cc];
                  ac[0] = fmaf(x, w0.x, ac[0]); ac[1] = fmaf(x, w0.y, ac[1]); ac[2] = fmaf(x, w0.z, ac[2]); ac[3] = fmaf(x, w0.w, ac[3]);
                  ac[4] = fmaf(x, w1.x, ac[4]); ac[5] = fmaf(x, w1.y, ac[5]); ac[6] = fmaf(x, w1.z, ac[6]); ac[7] = fmaf(x, w1.w, ac[7]);
                }
              }
        }
      }
    }
    uint4* outp = reinterpret_cast<uint4*>(p.out) + (size_t)n * (p.Cout >> 3) * P + v;
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      if (cc < (p.Cout >> 3) && active) {
        outp[(size_t)cc * P] = pack8<T>(acc[cc]);
#pragma unroll
        for (int q = 0; q < 8; ++q) { rs[cc * 8 + q] += acc[cc][q]; rq[cc * 8 + q] = fmaf(acc[cc][q], acc[cc][q], rq[cc * 8 + q]); }
      }
    }
  }
  // transposing butterfly: lane l ends with the warp total of channel l
#pragma unroll
  for (int k = 16; k >= 1; k >>= 1) {
    const bool up = (lane & k) != 0;
#pragma unroll
    for (int i = 0; i < k; ++i) {
      const float sa_ = up ? rs[i] : rs[i + k], ka_ = up ? rs[i + k] : rs[i];
      const float sb_ = up ? rq[i] : rq[i + k], kb_ = up ? rq[i + k] : rq[i];
      rs[i] = ka_ + __shfl_xor_sync(0xffffffffu, sa_, k);
      rq[i] = kb_ + __shfl_xor_sync(0xffffffffu, sb_, k);
    }
  }
  if (lane < p.Cout) { atomicAdd(&sstat[lane * 2], rs[0]); atomicAdd(&sstat[lane * 2 + 1], rq[0]); }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * p.Cout; c += blockDim.x)
    atomicAdd(p.sums + (size_t)n * p.Cout * 2 + c, (double)sstat[c]);
}

// ---------------------------------------------------------------------------------------------
// Generic direct conv on the chunked layout.  Block = 128 threads -> output tile 2(d) x 8(h) x 16(w),
// 32 output channels; thread = 2 w-adjacent voxels x 32 channels (64 fp32 accumulators).  Input
// channel chunks of 8 are staged with their halo in shared memory (16 B per voxel) next to the
// matching weight slice.  The input may be the channel concat of two tensors (decoder: up, skip).
// w packed: [Cin/8][Cout/32][taps][8 ci][32 co] fp32.
// ---------------------------------------------------------------------------------------------
struct ConvParams {
  const void* in0; int C0;
  const void* in1; int C1;
  const float* w;
  void* out;
  int out32;                   // raw output stored as fp32 [n][Cout/8][V][8] instead of T
  double* sums;
  int N, Di, Hi, Wi, Do, Ho, Wo, Cout;
  int kd, kh, kw, sd, sh, sw;
};
constexpr int GC_TD = 2, GC_TH = 8, GC_TW = 16, GC_COB = 32;

template <typename T>
__global__ void __launch_bounds__(128) conv_generic_kernel(ConvParams p) {
  extern __shared__ __align__(16) unsigned char smraw[];
  const int taps = p.kd * p.kh * p.kw;
  const int ed = (GC_TD - 1) * p.sd + p.kd, eh = (GC_TH - 1) * p.sh + p.kh, ew = (GC_TW - 1) * p.sw + p.kw;
  const int nin = ed * eh * ew;
  uint4* sin = reinterpret_cast<uint4*>(smraw);
  float* swt = reinterpret_cast<float*>(smraw + (size_t)nin * 16);
  __shared__ float sstat[GC_COB * 2];

  const int tiles_w = (p.Wo + GC_TW - 1) / GC_TW, tiles_h = (p.Ho + GC_TH - 1) / GC_TH;
  int tile = blockIdx.x;
  const int tw0 = (tile % tiles_w) * GC_TW; tile /= tiles_w;
  const int th0 = (tile % tiles_h) * GC_TH; tile /= tiles_h;
  const int td0 = tile * GC_TD;
  const int cob = blockIdx.y, n = blockIdx.z;
  const int tid = threadIdx.x;
  const int tp = tid & 7, th = (tid >> 3) & 7, td = tid >> 6;
  const int pd = p.kd >> 1, ph = p.kh >> 1, pw = p.kw >> 1;
  const int id0 = td0 * p.sd - pd, ih0 = th0 * p.sh - ph, iw0 = tw0 * p.sw - pw;
  const int64_t Vi = (int64_t)p.Di * p.Hi * p.Wi;
  const int Cin = p.C0 + p.C1;

  float acc0[GC_COB], acc1[GC_COB];
#pragma unroll
  for (int q = 0; q < GC_COB; ++q) { acc0[q] = 0.f; acc1[q] = 0.f; }
  if (tid < GC_COB * 2) sstat[tid] = 0.f;

  for (int cc = 0; cc < (Cin >> 3); ++cc) {
    const uint4* src = (cc * 8 < p.C0)
        ? reinterpret_cast<const uint4*>(p.in0) + ((size_t)n * (p.C0 >> 3) + cc) * Vi
        : reinterpret_cast<const uint4*>(p.in1) + ((size_t)n * (p.C1 >> 3) + (cc - (p.C0 >> 3))) * Vi;
    __syncthreads();
    for (int e = tid; e < nin; e += 128) {
      const int c = e % ew, b = (e / ew) % eh, a = e / (ew * eh);
      const int d = id0 + a, h = ih0 + b, w = iw0 + c;
      uint4 val = make_uint4(0, 0, 0, 0);
      if (d >= 0 && d < p.Di && h >= 0 && h < p.Hi && w >= 0 && w < p.Wi)
        val = __ldg(src + ((size_t)d * p.Hi + h) * p.Wi + w);
      sin[e] = val;
    }
    const float4* wsrc = reinterpret_cast<const float4*>(p.w + ((size_t)cc * (p.Cout / GC_COB) + cob) * taps * 8 * GC_COB);
    for (int e = tid; e < taps * 8 * GC_COB / 4; e += 128) reinterpret_cast<float4*>(swt)[e] = __ldg(wsrc + e);
    __syncthreads();
    int t = 0;
    for (int a = 0; a < p.kd; ++a)
      for (int b = 0; b < p.kh; ++b)
        for (int c = 0; c < p.kw; ++c, ++t) {
          const int base = ((td * p.sd + a) * eh + (th * p.sh + b)) * ew + (2 * tp) * p.sw + c;
          float xa[8], xb[8];
          unpack8<T>(sin[base], xa);
          unpack8<T>(sin[base + p.sw], xb);
          const float* wt = swt + t * 8 * GC_COB;
#pragma unroll
          for (int ci = 0; ci < 8; ++ci) {
#pragma unroll
            for (int q = 0; q < GC_COB; q += 4) {
              const float4 w4 = *reinterpret_cast<const float4*>(wt + ci * GC_COB + q);
              acc0[q + 0] = fmaf(xa[ci], w4.x, acc0[q + 0]); acc1[q + 0] = fmaf(xb[ci], w4.x, acc1[q + 0]);
              acc0[q + 1] = fmaf(xa[ci], w4.y, acc0[q + 1]); acc1[q + 1] = fmaf(xb[ci], w4.y, acc1[q + 1]);
              acc0[q + 2] = fmaf(xa[ci], w4.z, acc0[q + 2]); acc1[q + 2] = fmaf(xb[ci], w4.z, acc1[q + 2]);
              acc0[q + 3] = fmaf(xa[ci], w4.w, acc0[q + 3]); acc1[q + 3] = fmaf(xb[ci], w4.w, acc1[q + 3]);
            }
          }
        }
  }
  // epilogue: store + statistics
  const int od = td0 + td, oh = th0 + th, ow = tw0 + 2 * tp;
  const bool ok0 = od < p.Do && oh < p.Ho && ow < p.Wo;
  const bool ok1 = od < p.Do && oh < p.Ho && (ow + 1) < p.Wo;
  const int64_t Vo = (int64_t)p.Do * p.Ho * p.Wo;
  const size_t obase = ((size_t)n * (p.Cout >> 3) + cob * (GC_COB >> 3)) * Vo + ((size_t)od * p.Ho + oh) * p.Wo + ow;
  if (p.out32) {
    float4* o32 = reinterpret_cast<float4*>(p.out);
#pragma unroll
    for (int q8 = 0; q8 < GC_COB / 8; ++q8) {
      const size_t e = (obase + (size_t)q8 * Vo) * 2;
      if (ok0) { o32[e] = make_float4(acc0[q8 * 8], acc0[q8 * 8 + 1], acc0[q8 * 8 + 2], acc0[q8 * 8 + 3]); o32[e + 1] = make_float4(acc0[q8 * 8 + 4], acc0[q8 * 8 + 5], acc0[q8 * 8 + 6], acc0[q8 * 8 + 7]); }
      if (ok1) { o32[e + 2] = make_float4(acc1[q8 * 8], acc1[q8 * 8 + 1], acc1[q8 * 8 + 2], acc1[q8 * 8 + 3]); o32[e + 3] = make_float4(acc1[q8 * 8 + 4], acc1[q8 * 8 + 5], acc1[q8 * 8 + 6], acc1[q8 * 8 + 7]); }
    }
  } else {
    uint4* outp = reinterpret_cast<uint4*>(p.out) + obase;
#pragma unroll
    for (int q8 = 0; q8 < GC_COB / 8; ++q8) {
      if (ok0) outp[(size_t)q8 * Vo] = pack8<T>(acc0 + q8 * 8);
      if (ok1) outp[(size_t)q8 * Vo + 1] = pack8<T>(acc1 + q8 * 8);
    }
  }
  const int lane = tid & 31;
#pragma unroll
  for (int q = 0; q < GC_COB; ++q) {
    const float a = ok0 ? acc0[q] : 0.f, b = ok1 ? acc1[q] : 0.f;
    const float s = warp_sum(a + b), ss = warp_sum(a * a + b * b);
    if (lane == 0) { atomicAdd(&sstat[q * 2], s); atomicAdd(&sstat[q * 2 + 1], ss); }
  }
  __syncthreads();
  if (tid < GC_COB * 2) atomicAdd(p.sums + ((size_t)n * p.Cout + cob * GC_COB) * 2 + tid, (double)sstat[tid]);
}

// ---------------------------------------------------------------------------------------------
// InstanceNorm (instance statistics, biased variance, eps 1e-5, affine) + LeakyReLU(0.01), in place
// on the raw conv output.  grid.y = n * C/8 + chunk; coefficients computed once per block.
// ---------------------------------------------------------------------------------------------
// Optional second output: the parity-split ("space to depth") copy a strided tcgen05 conv consumes,
// s2d[n][class][C/8][D/sd][H/sh][W/sw][8] with class order tc_s2d_class().
struct S2dParams { void* dst; int D, H, W, sd, sh, sw; };

// QUAD: the four-voxel path for passes that also write a W-halving parity-split copy (a kernel of its own: with both paths in
// one kernel the extra registers of the quad path cost the plain passes 8 % of their bandwidth).
template <typename T, bool QUAD = false>
// raw and y alias when the layer is normalised in place (fp16 raw storage): no __restrict__ on either.
__global__ void __launch_bounds__(256) instnorm_lrelu_kernel(const void* raw, int raw32, void* y, NormParams np,
                                                             int C, int64_t V, S2dParams sp) {
  __shared__ float sa[8], sb[8];
  const int n = blockIdx.y / (C >> 3), cc = blockIdx.y % (C >> 3);
  if (threadIdx.x < 8) { float a, b; norm_coeffs(np, n, C, cc * 8 + threadIdx.x, a, b); sa[threadIdx.x] = a; sb[threadIdx.x] = b; }
  __syncthreads();
  float a[8], b[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { a[j] = sa[j]; b[j] = sb[j]; }
  uint4* row = reinterpret_cast<uint4*>(y) + (size_t)blockIdx.y * V;
  const uint4* rrow = reinterpret_cast<const uint4*>(raw) + (size_t)blockIdx.y * V;
  const float4* rrow32 = reinterpret_cast<const float4*>(raw) + (size_t)blockIdx.y * V * 2;
  const int nclass = sp.sd * sp.sh * sp.sw;
  const int Ds = sp.D / sp.sd, Hs = sp.H / sp.sh, Ws = sp.W / sp.sw;
  const int64_t Vs = (int64_t)Ds * Hs * Ws;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  auto s2d_store = [&](int64_t v, const uint4& o) {
    const int w = (int)(v % sp.W), h = (int)((v / sp.W) % sp.H), d = (int)(v / ((int64_t)sp.W * sp.H));
    const int c = tc_s2d_class(d, h, w, sp.sd, sp.sh, sp.sw);
    const int64_t vs = ((int64_t)(d / sp.sd) * Hs + (h / sp.sh)) * Ws + (w / sp.sw);
    reinterpret_cast<uint4*>(sp.dst)[(((size_t)n * nclass + c) * (C >> 3) + cc) * Vs + vs] = o;
  };
  if constexpr (QUAD) {
    // (launched only when sp.dst != nullptr, sp.sw == 2 and W % 4 == 0.)  Four consecutive voxels of a row per thread when the parity-split copy is written with W-halving: voxels 0, 2 go to one
    // class and 1, 3 to the next, each pair to adjacent slots, so the copy is written with 256-bit stores like the tensor itself
    // (with one 16-byte store per voxel these passes ran at 5.1 TB/s against 6.3 TB/s for the passes without a second output).
    const int64_t V4q = V >> 2;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < V4q; q += stride) {
      float f[4][8];
      if (raw32) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          uint4 q0, q1;
          ld_global_256(rrow32 + 8 * q + 2 * e, q0, q1);
          f[e][0] = __uint_as_float(q0.x); f[e][1] = __uint_as_float(q0.y); f[e][2] = __uint_as_float(q0.z); f[e][3] = __uint_as_float(q0.w);
          f[e][4] = __uint_as_float(q1.x); f[e][5] = __uint_as_float(q1.y); f[e][6] = __uint_as_float(q1.z); f[e][7] = __uint_as_float(q1.w);
        }
      } else {
        uint4 q0, q1, q2, q3;
        ld_global_256(rrow + 4 * q, q0, q1);
        ld_global_256(rrow + 4 * q + 2, q2, q3);
        unpack8<T>(q0, f[0]); unpack8<T>(q1, f[1]); unpack8<T>(q2, f[2]); unpack8<T>(q3, f[3]);
      }
      uint4 o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
#pragma unroll
        for (int j = 0; j < 8; ++j) f[e][j] = lrelu(fmaf(a[j], f[e][j], b[j]));
        o[e] = pack8<T>(f[e]);
      }
      st_global_256(row + 4 * q, o[0], o[1]);
      st_global_256(row + 4 * q + 2, o[2], o[3]);
      const int64_t v = 4 * q;
      const int w = (int)(v % sp.W), h = (int)((v / sp.W) % sp.H), d = (int)(v / ((int64_t)sp.W * sp.H));
      const int c0 = tc_s2d_class(d, h, w, sp.sd, sp.sh, sp.sw);                 // w even: the class of voxels 0, 2; voxels 1, 3: c0 + 1
      const int64_t vs = ((int64_t)(d / sp.sd) * Hs + (h / sp.sh)) * Ws + (w >> 1);
      uint4* d0 = reinterpret_cast<uint4*>(sp.dst) + (((size_t)n * nclass + c0) * (C >> 3) + cc) * Vs + vs;
      st_global_256(d0, o[0], o[2]);
      st_global_256(d0 + (size_t)(C >> 3) * Vs, o[1], o[3]);
    }
    return;
  } else {
  if ((V & 1) == 0) {
    // voxel pairs: one 256-bit load (fp16 raw) or two (fp32 raw), one 256-bit store
    const int64_t V2 = V >> 1;
    for (int64_t v2 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v2 < V2; v2 += stride) {
      float f[2][8];
      if (raw32) {
        uint4 q0, q1, q2, q3;
        ld_global_256(rrow32 + 4 * v2, q0, q1);
        ld_global_256(rrow32 + 4 * v2 + 2, q2, q3);
        const uint4 q[4] = {q0, q1, q2, q3};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          f[e][0] = __uint_as_float(q[2 * e].x); f[e][1] = __uint_as_float(q[2 * e].y); f[e][2] = __uint_as_float(q[2 * e].z); f[e][3] = __uint_as_float(q[2 * e].w);
          f[e][4] = __uint_as_float(q[2 * e + 1].x); f[e][5] = __uint_as_float(q[2 * e + 1].y); f[e][6] = __uint_as_float(q[2 * e + 1].z); f[e][7] = __uint_as_float(q[2 * e + 1].w);
        }
      } else {
        uint4 q0, q1;
        ld_global_256(rrow + 2 * v2, q0, q1);
        unpack8<T>(q0, f[0]); unpack8<T>(q1, f[1]);
      }
#pragma unroll
      for (int e = 0; e < 2; ++e)
#pragma unroll
        for (int j = 0; j < 8; ++j) f[e][j] = lrelu(fmaf(a[j], f[e][j], b[j]));
      const uint4 o0 = pack8<T>(f[0]), o1 = pack8<T>(f[1]);
      st_global_256(row + 2 * v2, o0, o1);
      if (sp.dst) { s2d_store(2 * v2, o0); s2d_store(2 * v2 + 1, o1); }
    }
    return;
  }
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += stride) {
    float f[8];
    if (raw32) {
      const float4 lo = rrow32[2 * v], hi = rrow32[2 * v + 1];
      f[0] = lo.x; f[1] = lo.y; f[2] = lo.z; f[3] = lo.w; f[4] = hi.x; f[5] = hi.y; f[6] = hi.z; f[7] = hi.w;
    } else unpack8<T>(rrow[v], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = lrelu(fmaf(a[j], f[j], b[j]));
    const uint4 o = pack8<T>(f);
    row[v] = o;
    if (sp.dst) s2d_store(v, o);
  }
  }   // !QUAD
}

// ---------------------------------------------------------------------------------------------
// Transposed conv with kernel == stride (each 1 or 2), bias-free (tu[u]).  Block = 128 input
// voxels x 32 output channels; loops over the kd*kh*kw taps, each tap writing one output parity.
// w packed: [Cout/32][taps][Cin][32 co] fp32.
// ---------------------------------------------------------------------------------------------
struct TConvParams {
  const void* in; void* out; const float* w;
  int N, Cin, Cout, Di, Hi, Wi, sd, sh, sw;
};

template <typename T>
__global__ void __launch_bounds__(128) tconv_kernel(TConvParams p) {
  extern __shared__ __align__(16) float swt[];          // [Cin][32]
  const int taps = p.sd * p.sh * p.sw;
  const int64_t Vi = (int64_t)p.Di * p.Hi * p.Wi;
  const int Do = p.Di * p.sd, Ho = p.Hi * p.sh, Wo = p.Wi * p.sw;
  const int64_t Vo = (int64_t)Do * Ho * Wo;
  const int cob = blockIdx.y, n = blockIdx.z;
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = v < Vi;
  const int w = (int)(v % p.Wi), h = (int)((v / p.Wi) % p.Hi), d = (int)(v / ((int64_t)p.Wi * p.Hi));
  const uint4* src = reinterpret_cast<const uint4*>(p.in) + (size_t)n * (p.Cin >> 3) * Vi + v;
  for (int t = 0; t < taps; ++t) {
    __syncthreads();
    const float4* wsrc = reinterpret_cast<const float4*>(p.w + ((size_t)cob * taps + t) * p.Cin * GC_COB);
    for (int e = threadIdx.x; e < p.Cin * GC_COB / 4; e += 128) reinterpret_cast<float4*>(swt)[e] = __ldg(wsrc + e);
    __syncthreads();
    float acc[GC_COB];
#pragma unroll
    for (int q = 0; q < GC_COB; ++q) acc[q] = 0.f;
    if (active) {
      for (int cc = 0; cc < (p.Cin >> 3); ++cc) {
        float x[8];
        unpack8<T>(__ldg(src + (size_t)cc * Vi), x);
#pragma unroll
        for (int ci = 0; ci < 8; ++ci) {
          const float* wt = swt + (cc * 8 + ci) * GC_COB;
#pragma unroll
          for (int q = 0; q < GC_COB; q += 4) {
            const float4 w4 = *reinterpret_cast<const float4*>(wt + q);
            acc[q + 0] = fmaf(x[ci], w4.x, acc[q + 0]); acc[q + 1] = fmaf(x[ci], w4.y, acc[q + 1]);
            acc[q + 2] = fmaf(x[ci], w4.z, acc[q + 2]); acc[q + 3] = fmaf(x[ci], w4.w, acc[q + 3]);
          }
        }
      }
      const int c = t % p.sw, b = (t / p.sw) % p.sh, a = t / (p.sw * p.sh);
      uint4* outp = reinterpret_cast<uint4*>(p.out) + ((size_t)n * (p.Cout >> 3) + cob * (GC_COB >> 3)) * Vo +
                    ((size_t)(d * p.sd + a) * Ho + (h * p.sh + b)) * Wo + (w * p.sw + c);
#pragma unroll
      for (int q8 = 0; q8 < GC_COB / 8; ++q8) outp[(size_t)q8 * Vo] = pack8<T>(acc + q8 * 8);
    }
  }
}

}  // namespace dwmh
