// conv3d 3x3x3 / stride 1 / pad 1 as a tcgen05 implicit GEMM (sm_100a), hand-written.
//
// GEMM view: M = output voxels, N = output channels, K = 27 taps x Cin.  One CTA owns a 16(H) x 8(W)
// output tile (128 GEMM rows = one UMMA_M) of one sample and one block of CB output channels and
// MARCHES ALONG D (the slowest spatial axis):
//   * TMA loads one haloed input plane chunk [KC/8][18][10][8ch] per step (x/y halo by TMA OOB zero
//     fill, the D halo by skipping out-of-range planes).  The chunked HBM layout makes the box land in
//     shared memory directly as a K-major, no-swizzle UMMA operand: 16 B per (voxel, 8-channel chunk),
//     SBO = 160 B between the 8-voxel rows, LBO = 2880 B between channel chunks.  The 9 in-plane taps
//     are 9 start addresses into the same plane (dy*160 + dx*16): each input byte is read from L2 once
//     and reused 27 x CB times from shared memory.
//   * the three D-taps are STACKED ALONG N: input plane d feeds output planes d-1, d, d+1, whose fp32
//     accumulators sit in neighbouring TMEM column blocks, so one tcgen05.mma of N = 3*CB consumes an
//     A window once for three taps (narrow layers, Cout = 32, would otherwise be bound by the
//     128 B/clk shared-memory operand bandwidth at ~40 % of the tensor peak).
//   * accumulators form a ring of R = 512/CB TMEM slots; the first MMA into an output plane overwrites
//     its slot (accumulate = 0), the later ones accumulate.  The epilogue warps drain a finished plane
//     (tcgen05.ld -> fp16/bf16 pack -> coalesced 16-B stores, InstanceNorm Welford partials (count,
//     mean, M2) per warp, merged in fp64 by stats_reduce_kernel) and hand the slot back.
//   * weights are pre-packed on the host as ready-made K-major operand tiles [kc][tap_yx][k8][3*CB][8]
//     and either stay resident in shared memory for the whole CTA or stream through a ring of bulk
//     copies.
// Warp roles of a group: 0 = TMA producer (activations), 1 = MMA issuer, 2..5 = epilogue, 6 = bulk-copy
// producer (weights); the norm-on-load kernels load through roles 0, 6, 7 and the first-conv kernels
// build their operand in roles 0, 6 with role 7 fetching input slices.  Which hardware warp takes which
// role is set by the kRole / kGroup tables in the kernel (epilogue warps first, issuers last); warp 1
// of the CTA allocates TMEM.  All hand-offs are mbarriers; nothing spins on __syncthreads.
#pragma once
#include <cuda.h>
#include <algorithm>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>
#include "common.cuh"
#include "tc_primitives.cuh"

namespace dwmh {

constexpr int TC_WARPS_PER_GROUP = 7;
constexpr int TC_THREADS = 224;          // per group; a dual-group CTA has 448
constexpr int TC_TH = 16, TC_TW = 8;
constexpr int TC_PH = 18, TC_PW = 10;
constexpr int TC_PLANE_BYTES = TC_PH * TC_PW * 16;     // one 8-channel chunk of a haloed plane
constexpr int TC_MAX_SA = 4, TC_MAX_NB = 40, TC_MAX_R = 16;
constexpr int TC_SMEM_MAX = 232448;                    // 227 KB opt-in limit
constexpr int TC_SMEM_RESERVED = 5120;                 // barriers + TMEM pointer + statistics
constexpr int TC_SMEM_RESERVED_FIRST = 10240;          // FIRST kernels: + two 4-slot rings of haloed input slices
constexpr int TC_FIRST_PITCH = 12;                     // words per ring row (10 used): 2 rows apart = 24 words -> conflict-free LDS
constexpr int TC_FIRST_SLICE = TC_PH * TC_FIRST_PITCH;
constexpr int TC_FIRST_STAGE_BYTES = 8 * 128 * 16;     // im2col operand of one output plane: 4 hi + 4 lo chunks of 8 taps

// One parity class of a strided conv (a plain stride-1 conv has exactly one class).  The producer tensor of
// a strided conv is stored a second time parity-split ("space to depth": [n][class][C/8][D/sd][H/sh][W/sw][8]),
// so a strided tap is again a dense TMA box plus a start-address shift.  tapmask: bit (dy*3+dx) = in-plane
// shifts this class uses; the sub-plane t of this class feeds output planes t+jlo .. t+jlo+jcnt-1.
struct TcClassDesc { int tapmask, jlo, jcnt, tile0; };

struct TcKParams {
  const void* wpack; void* out; StatPartial* partials;   // partials: [item][CB] (count, mean, M2)
  int C0, C1, Cout, CB, KC, nkc, nkc0;
  int nclass, Jlo, Jhi, jmax, tiles_per_kc, Din;
  int out32;                                 // raw output stored as fp32 instead of T
  int s222;                                  // stride (2,2,2): the standard 8 parity classes (straight-line issue path)
  int tconv, CBt, osd, osh, osw, Cout_t;   // transposed-conv mode: CB = osd*osh*osw * CBt, scatter epilogue
  TcClassDesc cls[8];
  int D, H, W, tilesH, tilesW, ZB, nzb, ncb;
  int SA, NB, resident, R, fmt;
  // norm-on-load (XFORM kernels): the input tensor is the producer's RAW fp16 output; three loader warps per group read each
  // plane from global memory into registers, apply InstanceNorm + LeakyReLU of the producer and store it into the activation stage
  const double* xf_sums; const float* xf_gamma; const float* xf_beta; double xf_inv_count; int xform; const void* xf_src;
  // FIRST kernels (first conv, 3x3x3): loader warps build an im2col operand from the fp32 volume / patches
  const float* fc_src; const SampleMeta* fc_metas; int fc_patch_mode, fc_SY, fc_SZ, first;
  int G;              // work-item pipelines ("groups") per CTA: 2 = two tiles share the resident weights, each with 256 TMEM columns
  int total_items;
  uint32_t a_stage_bytes, b_tile_bytes, off_b, off_bar;
  // multi-modality FIRST kernels (MULTI): fc_M input channels fc_mstride floats apart; the slice-ring barriers sit fc_sbar bytes
  // after off_bar (256 bytes per group)
  int fc_M; uint32_t fc_sbar; int64_t fc_mstride;
};

// Ordered second stage: every (sample, channel) combines the partials of its work items in index order, in fp64.
// partials: [item][CB]; the items of (n, cb) are the contiguous range [(n*ncb + cb) * ipb, +ipb).
// grid = nb * ncb blocks of CB * jn threads (c fastest -> coalesced 16-byte reads); out = {mean, biased variance}.
__global__ void __launch_bounds__(256) stats_reduce_kernel(const StatPartial* __restrict__ partials, double* __restrict__ out,
                                                           int ncb, int CB, int Cout, int ipb, int jn) {
  __shared__ double sh[3][256];
  const int n = blockIdx.x / ncb, cb = blockIdx.x % ncb;
  const int c = threadIdx.x % CB, j = threadIdx.x / CB;
  const StatPartial* base = partials + (size_t)blockIdx.x * ipb * CB + c;
  double cn = 0.0, cm = 0.0, cq = 0.0;
  for (int p = j; p < ipb; p += jn) {
    const float4 v = *reinterpret_cast<const float4*>(base + (size_t)p * CB);
    stat_merge<double>(cn, cm, cq, (double)v.x, (double)v.y, (double)v.z);
  }
  sh[0][threadIdx.x] = cn; sh[1][threadIdx.x] = cm; sh[2][threadIdx.x] = cq;
  __syncthreads();
  if (j == 0) {
    for (int jj = 1; jj < jn; ++jj) stat_merge<double>(cn, cm, cq, sh[0][jj * CB + c], sh[1][jj * CB + c], sh[2][jj * CB + c]);
    double* o = out + ((size_t)n * Cout + (size_t)cb * CB + c) * 2;
    o[0] = cm;
    o[1] = cn > 0.0 ? cq / cn : 0.0;
  }
}

// Ring-buffer cursor without div/mod.
struct RingPos {
  uint32_t idx = 0, phase = 0;
  __device__ __forceinline__ void advance(uint32_t n) { if (++idx == n) { idx = 0; phase ^= 1; } }
  __device__ __forceinline__ RingPos next(uint32_t n) const { RingPos r = *this; r.advance(n); return r; }
};

__device__ __forceinline__ uint64_t tc_desc(uint32_t hi, uint32_t lo) { return ((uint64_t)hi << 32) | lo; }

// start-address shift (16-byte units) of in-plane tap sft = dy*3 + dx inside a haloed 18 x 10 plane, 5 bits per tap
constexpr uint64_t tc_tap_shift_table() {
  uint64_t v = 0;
  for (int sft = 0; sft < 9; ++sft) v |= (uint64_t)((sft / 3) * TC_PW + (sft % 3)) << (5 * sft);
  return v;
}
constexpr uint64_t kTapShift = tc_tap_shift_table();

// KSTEPS = KC/16 (UMMA K steps per channel chunk); SMALL_CB: CB <= 32 -> per-thread running statistics.
// MULTI (FIRST only): p.fc_M > 1 input modalities, each plane is fc_M im2col stages accumulated into one TMEM slot.
template <typename T, int KSTEPS, bool SMALL_CB, bool TCONV, bool DUAL, bool XFORM, bool FIRST = false, bool MULTI = false>
__global__ void __launch_bounds__((DUAL ? 2 : 1) * (TC_THREADS + ((FIRST || XFORM) ? 32 : 0)), 1)
conv3_tc_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1, const TcKParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = tc::smem_u32(smem);
  const int warp_abs = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Dual-group CTA: two independent tile pipelines (own activation ring, accumulator ring, warps) share the
  // resident weight tiles; while one group's issue thread sits in barrier latency or bookkeeping the other
  // group's MMAs keep the tensor pipe busy.
  constexpr int WPG = TC_WARPS_PER_GROUP;
  constexpr int TPG = WPG * 32;
  constexpr int NG = DUAL ? 2 : 1;
  // role: 0 act producer, 1 MMA, 2..5 epilogue, 6 weight producer (+ transform in XFORM kernels), 7 slice fetcher (FIRST) / transform (XFORM).
  // Warp numbering: the epilogue warps come first (TMEM lane quarter = warp_abs & 3 for both groups), the light producer warps next,
  // the MMA issuers last and on different schedulers (warp_abs % 4); each scheduler gets two epilogue warps and, in the 16-warp
  // kernels, one transform / builder warp.  (Measured against the original numbering -- issuer = warp 1 of each group, two transform
  // warps on one scheduler -- and against issuer bookkeeping without tcgen05 fences / barrier peeks: all within +-1 % of 42.2 ms per
  // 32-forward batch, so the ~500-1200 cycles per plane the issuer spends outside its MMA bursts and timed waits are not a
  // scheduling artefact; DESIGN.md section 4.)
  constexpr bool EXTRA = FIRST || XFORM;
  int g, warp;
  if constexpr (!DUAL) {
    //            warp_abs:  0  1  2  3  4  5  6  7
    constexpr unsigned char kRole7[7] = {2, 3, 4, 5, 0, 6, 1};
    constexpr unsigned char kRole8[8] = {2, 3, 4, 5, 0, 6, 7, 1};
    g = 0; warp = EXTRA ? kRole8[warp_abs] : kRole7[warp_abs];
  } else if constexpr (!EXTRA) {
    //            warp_abs:   0  1  2  3  4  5  6  7  8  9 10 11 12 13
    constexpr unsigned char kGroup14[14] = {0, 0, 0, 0, 1, 1, 1, 1, 0, 1, 0, 1, 1, 0};
    constexpr unsigned char kRole14[14] = {2, 3, 4, 5, 2, 3, 4, 5, 0, 0, 6, 6, 1, 1};
    g = kGroup14[warp_abs]; warp = kRole14[warp_abs];
  } else {
    //            warp_abs:   0  1  2  3  4  5  6  7  8  9 10 11 12 13 14 15
    constexpr unsigned char kGroup16[16] = {0, 0, 0, 0, 1, 1, 1, 1, 0, 1, 1, 1, 0, 0, 1, 0};
    constexpr unsigned char kRole16[16] = {2, 3, 4, 5, 2, 3, 4, 5, 0, 0, 6, 7, 6, 7, 1, 1};
    g = kGroup16[warp_abs]; warp = kRole16[warp_abs];
  }
  const bool extra = warp == 7;

  int wi = blockIdx.x * p.G + g;
  const bool idle = wi >= p.total_items;
  if (idle) wi = p.total_items - 1;
  const int tw = wi % p.tilesW; wi /= p.tilesW;
  const int th = wi % p.tilesH; wi /= p.tilesH;
  const int zb = wi % p.nzb; wi /= p.nzb;
  const int cb = wi % p.ncb; wi /= p.ncb;
  const int n = wi;
  const int h0 = th * TC_TH, w0 = tw * TC_TW;
  const int z_lo = zb * p.ZB, z_end = min(p.D, z_lo + p.ZB);
  const uint32_t SA = p.SA, NB = p.NB, R = p.R, CB = p.CB;

  const uint32_t nbar = 3 * SA + 2 * NB + 2 * R;      // a_full, a_empty, b_full, b_empty, acc_full, acc_empty, a_ready
  const uint32_t bar0 = smem_base + p.off_bar, bar = bar0 + (uint32_t)g * nbar * 8u;
  const uint32_t a_full = bar, a_empty = bar + 8u * SA;
  const uint32_t b_full = bar0 + 16u * SA, b_empty = b_full + 8u * NB;             // weight ring: shared, lives in group 0's block
  const uint32_t acc_full = bar + 16u * SA + 16u * NB, acc_empty = acc_full + 8u * R;
  const uint32_t a_ready = acc_empty + 8u * R;          // XFORM: plane transformed, ready for the MMA
  const uint32_t a_mma = (XFORM || FIRST) ? a_ready : a_full;      // what the MMA issuer waits on
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem + p.off_bar + 8 * nbar * p.G);
  const uint32_t aux_off = (p.off_bar + 8u * nbar * (uint32_t)p.G + 16u + 8u) & ~15u;      // 16-byte aligned (the loaders read coefficients as float4)
  float* s_coef = reinterpret_cast<float*>(smem + aux_off) + (size_t)p.G * 2 * CB + (size_t)g * 2 * 64;   // XFORM: a[64], b[64]
  // FIRST: ring of haloed input slices, 4 slots (MULTI: 4 per modality)
  const int NM = MULTI ? p.fc_M : 1;
  float* s_slice = reinterpret_cast<float*>(smem + aux_off) + (size_t)p.G * 2 * CB + (size_t)p.G * 2 * 64 + (size_t)g * 4 * NM * TC_FIRST_SLICE;
  const uint32_t smem_a = smem_base + (uint32_t)g * SA * p.a_stage_bytes;          // this group's activation ring
  // UMMA shared-memory descriptors hold a 14-bit (address >> 4): descriptor arithmetic uses the masked offsets
  const uint32_t smem_a_d = smem_a & 0x3FFFFu, smem_b_d = (smem_base + p.off_b) & 0x3FFFFu;
  // FIRST: slice ring barriers (MULTI: up to 16 slots of each kind per group)
  const uint32_t s_full = MULTI ? smem_base + p.off_bar + p.fc_sbar + (uint32_t)g * 256u
                                : smem_base + p.off_bar + TC_SMEM_RESERVED_FIRST - 128 + (uint32_t)g * 64u;
  const uint32_t s_empty = s_full + (MULTI ? 128u : 32u);

  if (threadIdx.x == 0) {
    if constexpr (!FIRST) {
      tc::prefetch_tensormap(&tmA0);
      tc::prefetch_tensormap(&tmA1);
    }
    for (int gg = 0; gg < p.G; ++gg) {
      const uint32_t bg = bar0 + (uint32_t)gg * nbar * 8u;
      for (uint32_t s_ = 0; s_ < SA; ++s_) { tc::mbar_init(bg + 8 * s_, 1); tc::mbar_init(bg + 8 * (SA + s_), 1); }
      for (uint32_t s_ = 0; s_ < R; ++s_) { tc::mbar_init(bg + 16 * SA + 16 * NB + 8 * s_, 1); tc::mbar_init(bg + 16 * SA + 16 * NB + 8 * (R + s_), 4); }
      for (uint32_t s_ = 0; s_ < SA; ++s_) tc::mbar_init(bg + 16 * SA + 16 * NB + 16 * R + 8 * s_, XFORM ? 3 : 2);
    }
    if constexpr (FIRST && MULTI)
      for (int gg = 0; gg < p.G; ++gg)
        for (int s_ = 0; s_ < 4 * NM; ++s_) {
          tc::mbar_init(smem_base + p.off_bar + p.fc_sbar + gg * 256 + 8 * s_, 1);
          tc::mbar_init(smem_base + p.off_bar + p.fc_sbar + gg * 256 + 128 + 8 * s_, 2);
        }
    else if constexpr (FIRST)
      for (int gg = 0; gg < p.G; ++gg)
        for (uint32_t s_ = 0; s_ < 4; ++s_) {
          tc::mbar_init(smem_base + p.off_bar + TC_SMEM_RESERVED_FIRST - 128 + gg * 64 + 8 * s_, 1);
          tc::mbar_init(smem_base + p.off_bar + TC_SMEM_RESERVED_FIRST - 128 + gg * 64 + 32 + 8 * s_, 2);
        }
    const uint32_t nactive = (uint32_t)min(p.G, p.total_items - (int)blockIdx.x * p.G);      // groups of this CTA that have a tile
    for (uint32_t s_ = 0; s_ < NB; ++s_) { tc::mbar_init(b_full + 8 * s_, 1); tc::mbar_init(b_empty + 8 * s_, nactive); }
    tc::fence_barrier_init();
  }
  if (warp_abs == 1) tc::tmem_alloc(tc::smem_u32(tmem_ptr_smem), 512);
  if constexpr (XFORM) {
    // each group: coefficients of ITS sample
    for (int i = threadIdx.x; i < p.G * p.C0; i += blockDim.x) {
      const int gg = i / p.C0, c_ = i - gg * p.C0;
      const int item = min((int)blockIdx.x * p.G + gg, p.total_items - 1);
      const int n_gg = item / (p.tilesW * p.tilesH * p.nzb * p.ncb);
      NormParams np{p.xf_sums, p.xf_gamma, p.xf_beta, p.xf_inv_count};
      float a_, b_;
      norm_coeffs(np, n_gg, p.C0, c_, a_, b_);
      float* co = reinterpret_cast<float*>(smem + aux_off) + (size_t)p.G * 2 * CB + (size_t)gg * 2 * 64;
      co[c_] = a_; co[64 + c_] = b_;
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem + (uint32_t)g * 256u;       // group 1 owns TMEM columns 256..511

  if (idle) {
    // odd item count: the second group of the last CTA has nothing to do
  } else
  if (FIRST && MULTI && warp == 7) {
    // ---------------- multi-modality first conv: slice fetcher ---------------------------------------------------------
    // As below, for NM modalities: slice q = k * NM + m is plane z_lo - 1 + k of modality m, ring slot q % (4 NM).
    int ox = 0, oy = 0, oz = 0, flip = 0;
    const float* src = p.fc_src;
    int SY = p.fc_SY, SZ = p.fc_SZ;
    if (p.fc_patch_mode) { src += (size_t)n * NM * p.D * p.H * p.W; SY = p.H; SZ = p.W; }
    else { const SampleMeta m_ = p.fc_metas[n]; ox = m_.ox; oy = m_.oy; oz = m_.oz; flip = m_.flip; }
    int sgoff[6]; bool sin_[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const int pos = lane + 32 * i;
      const int r = pos / TC_PW, c = pos - r * TC_PW;
      const int hh = h0 - 1 + r, ww = w0 - 1 + c;
      sin_[i] = pos < TC_PH * TC_PW && (unsigned)hh < (unsigned)p.H && (unsigned)ww < (unsigned)p.W;
      const int sj = oy + ((flip & 2) ? p.H - 1 - hh : hh), sk = oz + ((flip & 1) ? p.W - 1 - ww : ww);
      sgoff[i] = sin_[i] ? sj * SZ + sk : 0;
    }
    const float* sbase = src + (size_t)ox * SY * SZ;
    const int zstep = (flip & 4) ? -SY * SZ : SY * SZ;
    if (flip & 4) sbase += (size_t)(p.D - 1) * SY * SZ;
    const int nq = (z_end - z_lo + 2) * NM, RS = 4 * NM;
    constexpr uint32_t kHiMask = ActT<T>::kUmmaFormat == 0 ? 0xFFFFE000u : 0xFFFF0000u;
    uint32_t* ring = reinterpret_cast<uint32_t*>(s_slice);
    auto fetch = [&](int q, float v[6]) {
      const int k = q / NM, m = q - k * NM;
      const int zz = z_lo - 1 + k;
      const bool zin = q < nq && (unsigned)zz < (unsigned)p.D;
      const float* sp = sbase + (ptrdiff_t)m * p.fc_mstride + (ptrdiff_t)zz * zstep;
#pragma unroll
      for (int i = 0; i < 6; ++i) v[i] = (zin && sin_[i]) ? __ldg(sp + sgoff[i]) : 0.f;
    };
    auto step = [&](int q, float (&v)[6]) {
      const int slot = q % RS;
      if (q >= RS) tc::mbar_wait(s_empty + 8 * slot, ((q / RS) & 1) ^ 1, 10);
      uint32_t* dst = ring + slot * TC_FIRST_SLICE;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const float hf = __uint_as_float(__float_as_uint(v[i]) & kHiMask);
        const int pos = lane + 32 * i, r = pos / TC_PW;
        if (pos < TC_PH * TC_PW) dst[r * TC_FIRST_PITCH + (pos - r * TC_PW)] = ActT<T>::from_f2(hf, v[i] - hf);
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(s_full + 8 * slot);
      fetch(q + 4, v);
    };
    float v0[6], v1[6], v2[6], v3[6];
    fetch(0, v0); fetch(1, v1); fetch(2, v2); fetch(3, v3);
    for (int q = 0; q < nq; q += 4) {
      step(q, v0);
      if (q + 1 < nq) step(q + 1, v1);
      if (q + 2 < nq) step(q + 2, v2);
      if (q + 3 < nq) step(q + 3, v3);
    }
  } else if (FIRST && MULTI && (warp == 0 || warp == 6)) {
    // ---------------- multi-modality first conv: builder warps -----------------------------------------------------------
    // One im2col stage per (plane, modality), built exactly as below from that modality's three slices; the MMA issuer
    // accumulates the NM stages of a plane into one TMEM slot.
    const bool leader = tc::elect_one();
    if (warp == 6 && g == 0 && leader) {
      tc::mbar_arrive_expect_tx(b_full, p.b_tile_bytes);
      tc::bulk_load(smem_base + p.off_b, p.wpack, p.b_tile_bytes, b_full);
    }
    const int l64 = (warp == 0 ? 0 : 32) + lane;
    const uint32_t* ring = reinterpret_cast<const uint32_t*>(s_slice);
    const int RS = 4 * NM;
    for (int q = 0; q < 2 * NM; ++q) tc::mbar_wait(s_full + 8 * q, 0, 11);
    RingPos xf;
    for (int j = 0; j < z_end - z_lo; ++j) {
      for (int m = 0; m < NM; ++m) {
        const int q2 = (j + 2) * NM + m;
        tc::mbar_wait(s_full + 8 * (q2 % RS), (q2 / RS) & 1, 11);
        tc::mbar_wait(a_empty + 8 * xf.idx, xf.phase ^ 1, 9);
        uint4* stage = reinterpret_cast<uint4*>(smem + (size_t)g * SA * p.a_stage_bytes + (size_t)xf.idx * p.a_stage_bytes);
        const uint32_t* sl[3] = {ring + ((j * NM + m) % RS) * TC_FIRST_SLICE, ring + (((j + 1) * NM + m) % RS) * TC_FIRST_SLICE,
                                 ring + (q2 % RS) * TC_FIRST_SLICE};
        const int hh = (l64 >> 3) * 2, ww = l64 & 7;
        uint32_t val[3][4][3];
#pragma unroll
        for (int dz = 0; dz < 3; ++dz)
#pragma unroll
          for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) val[dz][r][kw] = sl[dz][(hh + r) * TC_FIRST_PITCH + ww + kw];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const int mrow = (hh + rr) * 8 + ww;
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            uint32_t x[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int tap = 2 * q + e;
              x[e] = tap < 27 ? val[tap / 9][(tap / 3) % 3 + rr][tap % 3] : 0u;
            }
            hi[q] = __byte_perm(x[0], x[1], 0x5410);
            lo[q] = __byte_perm(x[0], x[1], 0x7632);
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            stage[c * 128 + mrow] = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
            stage[(4 + c) * 128 + mrow] = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
          }
        }
        tc::fence_proxy_async();
        __syncwarp();
        if (lane == 0) { tc::mbar_arrive(a_ready + 8 * xf.idx); tc::mbar_arrive(s_empty + 8 * ((j * NM + m) % RS)); }
        xf.advance(SA);
      }
    }
  } else
  if (FIRST && warp == 7) {
    // ---------------- first conv (Cin = 1): slice fetcher (extra warps 14, 15 of the CTA) ------------
    // Streams the haloed 18 x 10 input slices of this tile (zero outside the patch, tile origin and mirror flip applied
    // to the source index) into a 4-slot ring, each value already split x = hi + lo: low half = hi (x truncated to the
    // 16-bit format, exact), high half = lo = rn(x - hi).  A warp of its own because the builders' proxy fence
    // (MEMBAR + FENCE.VIEW.ASYNC) waits for every outstanding global load of the executing warp: with the prefetch in
    // the builder warps each plane cost one full HBM latency.
    int ox = 0, oy = 0, oz = 0, flip = 0;
    const float* src = p.fc_src;
    int SY = p.fc_SY, SZ = p.fc_SZ;
    if (p.fc_patch_mode) { src += (size_t)n * p.D * p.H * p.W; SY = p.H; SZ = p.W; }
    else { const SampleMeta m_ = p.fc_metas[n]; ox = m_.ox; oy = m_.oy; oz = m_.oz; flip = m_.flip; }
    int sgoff[6]; bool sin_[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const int pos = lane + 32 * i;
      const int r = pos / TC_PW, c = pos - r * TC_PW;
      const int hh = h0 - 1 + r, ww = w0 - 1 + c;
      sin_[i] = pos < TC_PH * TC_PW && (unsigned)hh < (unsigned)p.H && (unsigned)ww < (unsigned)p.W;
      const int sj = oy + ((flip & 2) ? p.H - 1 - hh : hh), sk = oz + ((flip & 1) ? p.W - 1 - ww : ww);
      sgoff[i] = sin_[i] ? sj * SZ + sk : 0;
    }
    const float* sbase = src + (size_t)ox * SY * SZ;
    const int zstep = (flip & 4) ? -SY * SZ : SY * SZ;
    if (flip & 4) sbase += (size_t)(p.D - 1) * SY * SZ;
    const int nslices = z_end - z_lo + 2;                       // slice k = patch plane z_lo - 1 + k
    constexpr uint32_t kHiMask = ActT<T>::kUmmaFormat == 0 ? 0xFFFFE000u : 0xFFFF0000u;
    uint32_t* ring = reinterpret_cast<uint32_t*>(s_slice);
    auto fetch = [&](int k, float v[6]) {
      const int zz = z_lo - 1 + k;
      const bool zin = k < nslices && (unsigned)zz < (unsigned)p.D;
      const float* sp = sbase + (ptrdiff_t)zz * zstep;
#pragma unroll
      for (int i = 0; i < 6; ++i) v[i] = (zin && sin_[i]) ? __ldg(sp + sgoff[i]) : 0.f;
    };
    auto step = [&](int k, float (&v)[6]) {
      if (k >= 4) tc::mbar_wait(s_empty + 8 * (k & 3), ((k >> 2) & 1) ^ 1, 10);
      uint32_t* dst = ring + (k & 3) * TC_FIRST_SLICE;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const float hf = __uint_as_float(__float_as_uint(v[i]) & kHiMask);
        const int pos = lane + 32 * i, r = pos / TC_PW;
        if (pos < TC_PH * TC_PW) dst[r * TC_FIRST_PITCH + (pos - r * TC_PW)] = ActT<T>::from_f2(hf, v[i] - hf);
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(s_full + 8 * (k & 3));
      fetch(k + 4, v);                                          // HBM latency is several planes long: 4 slices in flight
    };
    float v0[6], v1[6], v2[6], v3[6];
    fetch(0, v0); fetch(1, v1); fetch(2, v2); fetch(3, v3);
    for (int k = 0; k < nslices; k += 4) {
      step(k, v0);
      if (k + 1 < nslices) step(k + 1, v1);
      if (k + 2 < nslices) step(k + 2, v2);
      if (k + 3 < nslices) step(k + 3, v3);
    }
  } else if (FIRST && (warp == 0 || warp == 6)) {
    // ---------------- first conv (Cin = 1): builder warps write the im2col operand -------------------
    // Row m of the operand = output voxel (h0 + m/8, w0 + m%8) of plane t, columns = its 27 neighbours (hi halves in
    // chunks 0..3, lo halves in chunks 4..7), so that x*w = hi*w_hi + lo*w_hi + hi*w_lo keeps fp32-level accuracy on
    // the tensor cores (K = 3 x 32).  Stage layout: [8 chunks][128 rows][16 B]  (K-major, SBO = 128 B, LBO = 2048 B).
    const bool leader = tc::elect_one();
    if (warp == 6 && g == 0 && leader) {
      tc::mbar_arrive_expect_tx(b_full, p.b_tile_bytes);
      tc::bulk_load(smem_base + p.off_b, p.wpack, p.b_tile_bytes, b_full);
    }
    const int l64 = (warp == 0 ? 0 : 32) + lane;
    const uint32_t* ring = reinterpret_cast<const uint32_t*>(s_slice);
    tc::mbar_wait(s_full, 0, 11);
    tc::mbar_wait(s_full + 8, 0, 11);
    RingPos xf;
    for (int j = 0; j < z_end - z_lo; ++j) {                    // plane t = z_lo + j reads slices j, j+1, j+2
      tc::mbar_wait(s_full + 8 * ((j + 2) & 3), ((j + 2) >> 2) & 1, 11);
      tc::mbar_wait(a_empty + 8 * xf.idx, xf.phase ^ 1, 9);
      uint4* stage = reinterpret_cast<uint4*>(smem + (size_t)g * SA * p.a_stage_bytes + (size_t)xf.idx * p.a_stage_bytes);
      const uint32_t* sl[3] = {ring + (j & 3) * TC_FIRST_SLICE, ring + ((j + 1) & 3) * TC_FIRST_SLICE, ring + ((j + 2) & 3) * TC_FIRST_SLICE};
      // a lane builds two vertically adjacent rows (hh, ww), (hh + 1, ww): they share 2 of their 3 input rows
      const int hh = (l64 >> 3) * 2, ww = l64 & 7;
      uint32_t val[3][4][3];
#pragma unroll
      for (int dz = 0; dz < 3; ++dz)
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) val[dz][r][kw] = sl[dz][(hh + r) * TC_FIRST_PITCH + ww + kw];
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const int m = (hh + rr) * 8 + ww;
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          uint32_t x[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int tap = 2 * q + e;
            x[e] = tap < 27 ? val[tap / 9][(tap / 3) % 3 + rr][tap % 3] : 0u;
          }
          hi[q] = __byte_perm(x[0], x[1], 0x5410);
          lo[q] = __byte_perm(x[0], x[1], 0x7632);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          stage[c * 128 + m] = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
          stage[(4 + c) * 128 + m] = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
        }
      }
      tc::fence_proxy_async();
      __syncwarp();
      if (lane == 0) { tc::mbar_arrive(a_ready + 8 * xf.idx); tc::mbar_arrive(s_empty + 8 * (j & 3)); }
      xf.advance(SA);
    }
  } else if (XFORM && (warp == 0 || warp == 6 || warp == 7)) {
    // ---------------- norm-on-load: three loader / transform warps per group (roles 0, 6, 7) -----------
    // (plain stride-1 layer, 32-channel chunks, <= 64 channels on load.)  The source is the producer layer's RAW fp16 output:
    // each lane streams its 16-byte slots of the haloed plane (one slot = 8 channels of one position) from global memory into
    // registers, applies InstanceNorm + LeakyReLU of the producer, writes the result into the activation stage (positions
    // outside the image stay exactly 0) and signals a_ready.  Shared-memory traffic per plane and group: one 11.5 KB write,
    // against TMA write + load + store (34.5 KB) of an in-place transform -- in a kernel whose MMAs are bound by shared-memory
    // operand reads.
    const bool leader = tc::elect_one();
    if (warp == 6 && g == 0 && leader) {
      const int ntile = p.nkc * p.tiles_per_kc;
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.wpack) + (size_t)cb * ntile * p.b_tile_bytes;
      for (int t = 0; t < ntile; ++t) {
        tc::mbar_arrive_expect_tx(b_full + 8 * t, p.b_tile_bytes);
        tc::bulk_load(smem_base + p.off_b + t * p.b_tile_bytes, wsrc + (size_t)t * p.b_tile_bytes, p.b_tile_bytes, b_full + 8 * t);
      }
    }
    // slots of one stage: [4 chunks][180 positions] of 16 bytes.  Every loader owns 60 positions of ALL four chunks: iteration i
    // handles chunk i / 2, positions 60 wl + 32 (i & 1) + lane (the odd iterations are 28 lanes wide), so the chunk -- hence the
    // coefficient set and the stage offset -- of an unrolled iteration is a compile-time constant and the three loaders run ONE
    // copy of the loop.  What this code is tuned for (ncu source-level sampling, DESIGN.md section 4):
    //   * instruction footprint: a version with one specialised copy per loader ran slower although it executed 40 % fewer
    //     instructions -- half of all samples of the loaders AND of the epilogue warps became instruction-fetch stalls
    //     (the roles of this kernel run five different code regions at once);
    //   * registers: 128 per thread in the 512-thread CTA, and a spill is an L2 round trip here (227 KB of the SM's 256 KB are
    //     carved out as shared memory: the L1 cannot hold 512 stack frames).  Load buffer 32, coefficients of ONE chunk 16
    //     (re-read from shared memory when the chunk changes, 4 x per plane), two position offsets;
    //   * scoreboards: ptxas puts all loads of the buffer on ONE scoreboard, so a wait for any slot is a wait for every load
    //     issued before it -- reloading slot by slot made each slot wait for the load issued one slot earlier.  The buffer is
    //     therefore reloaded as one batch after the last slot has left its registers; it lands while the warp writes that
    //     slot, signals, and waits for the next free stage.  (A TMA prefetch of the coming boxes into L2 changed nothing.)
    constexpr int NPOS = TC_PH * TC_PW, NIT = 8, PPW = NPOS / 3;      // 180 positions, 60 per loader
    const int wl = warp == 0 ? 0 : warp - 5;
    const int HW = p.H * p.W;
    const size_t V4 = (size_t)p.Din * HW;                   // 16-byte vectors per 8-channel chunk of one sample
    uint32_t poff[2];
    bool pin[2], pborder[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int pos = PPW * wl + 32 * k + lane;
      const int r = pos / TC_PW, c = pos - r * TC_PW;
      const int hh = h0 - 1 + r, ww = w0 - 1 + c;
      const bool v = 32 * k + lane < PPW;
      pin[k] = v && (unsigned)hh < (unsigned)p.H && (unsigned)ww < (unsigned)p.W;
      pborder[k] = v && !pin[k];                            // a slot of the stage that lies outside the image (stays 0)
      poff[k] = pin[k] ? (uint32_t)(hh * p.W + ww) : 0u;
    }
    const uint32_t slot0 = (uint32_t)(PPW * wl + lane) * 16u;
    // positions outside the image are written ONCE (zero) in every stage and never again: the tile, hence the set of such slots,
    // is the same for every plane of the CTA (planes outside the volume are skipped altogether)
    if (pborder[0] || pborder[1]) {
      for (uint32_t s_ = 0; s_ < SA; ++s_)
#pragma unroll
        for (int i = 0; i < NIT; ++i)
          if (pborder[i & 1]) st_shared_128(smem_a + s_ * p.a_stage_bytes + slot0 + ((i >> 1) * NPOS + 32 * (i & 1)) * 16, make_uint4(0u, 0u, 0u, 0u));
    }
    const uint4* src_n = reinterpret_cast<const uint4*>(p.xf_src) + (size_t)n * (p.C0 >> 3) * V4;
    const int t_last = min(z_end - 1 - p.Jlo, p.Din - 1), t_first = max(z_lo - p.Jhi, 0);
    int t_ld = t_first, kc_ld = 0;                           // next (plane, channel chunk) of the raw source to load
    auto next_src = [&]() -> const uint4* {
      if (t_ld > t_last) return nullptr;
      const uint4* sp = src_n + (size_t)(kc_ld * 4) * V4 + (size_t)t_ld * HW;
      if (++kc_ld == p.nkc) { kc_ld = 0; ++t_ld; }
      return sp;
    };
    RingPos xf;
    uint4 buf[NIT];
    {
      const uint4* sp = next_src();
      if (sp) {
#pragma unroll
        for (int i = 0; i < NIT; ++i) buf[i] = pin[i & 1] ? ld_stream(sp + (size_t)(i >> 1) * V4 + poff[i & 1]) : make_uint4(0u, 0u, 0u, 0u);
      }
    }
    for (int t_use = t_first; t_use <= t_last; ++t_use) {
      for (int kc_use = 0; kc_use < p.nkc; ++kc_use) {
        tc::mbar_wait(a_empty + 8 * xf.idx, xf.phase ^ 1, 8);
        const uint4* sp_next = next_src();
        uint32_t stage = smem_a + xf.idx * p.a_stage_bytes + slot0;        // 32-bit shared address, kept opaque so that it stays in ONE
        asm volatile("" : "+r"(stage));                                     // register (under pressure ptxas rebuilt it per slot from S2R / LDC chains)
        const float4* co4 = reinterpret_cast<const float4*>(s_coef + kc_use * 32);
        float ca[8], cb[8];
#pragma unroll
        for (int i = 0; i < NIT; ++i) {
          if ((i & 1) == 0) {                                   // coefficients of this iteration's chunk
            const float4 a_lo = co4[i], a_hi = co4[i + 1], b_lo = co4[16 + i], b_hi = co4[17 + i];
            ca[0] = a_lo.x; ca[1] = a_lo.y; ca[2] = a_lo.z; ca[3] = a_lo.w; ca[4] = a_hi.x; ca[5] = a_hi.y; ca[6] = a_hi.z; ca[7] = a_hi.w;
            cb[0] = b_lo.x; cb[1] = b_lo.y; cb[2] = b_lo.z; cb[3] = b_lo.w; cb[4] = b_hi.x; cb[5] = b_hi.y; cb[6] = b_hi.z; cb[7] = b_hi.w;
          }
          float f[8];
          unpack8<T>(buf[i], f);
          if (i == NIT - 1 && sp_next) {
#pragma unroll
            for (int q = 0; q < NIT; ++q)
              if (pin[q & 1]) buf[q] = ld_stream(sp_next + (size_t)(q >> 1) * V4 + poff[q & 1]);
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float z = fmaf(ca[e], f[e], cb[e]);
            f[e] = fmaxf(z, 0.01f * z);
          }
          if (pin[i & 1]) st_shared_128(stage + ((i >> 1) * NPOS + 32 * (i & 1)) * 16, pack8<T>(f));
        }
        tc::fence_proxy_async();          // generic-proxy stores -> async-proxy (UMMA) reads
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(a_ready + 8 * xf.idx);
        xf.advance(SA);
      }
    }
  } else if (warp == 0) {
    // ---------------- activation producer: one TMA box per (input plane, channel chunk) -----------
    const bool leader = tc::elect_one();
    RingPos a;
    for (int t = z_lo - p.Jhi; t <= z_end - 1 - p.Jlo; ++t) {
      if (t < 0 || t >= p.Din) continue;
      for (int c = 0; c < p.nclass; ++c) {
        if (max(t + p.cls[c].jlo, z_lo) > min(t + p.cls[c].jlo + p.cls[c].jcnt - 1, z_end - 1)) continue;
        for (int kc = 0; kc < p.nkc; ++kc) {
          tc::mbar_wait(a_empty + 8 * a.idx, a.phase ^ 1, 1);
          if (leader) {
            tc::mbar_arrive_expect_tx(a_full + 8 * a.idx, p.a_stage_bytes);
            const bool first = kc < p.nkc0;
            const int c8 = first ? (n * p.nclass + c) * (p.C0 >> 3) + kc * (2 * KSTEPS) : n * (p.C1 >> 3) + (kc - p.nkc0) * (2 * KSTEPS);
            tc::tma_load_4d(smem_a + a.idx * p.a_stage_bytes, first ? &tmA0 : &tmA1, a_full + 8 * a.idx, (w0 - 1) * 8, h0 - 1, t, c8);
          }
          a.advance(SA);
        }
      }
    }
  } else if (warp == 6) {
    // ---------------- weight producer: ready-made operand tiles, bulk copies ----------------------
    const bool leader = tc::elect_one();
    const int ntile = p.nkc * p.tiles_per_kc;
    const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.wpack) + (size_t)cb * ntile * p.b_tile_bytes;
    if (p.resident) {
      if (leader && g == 0)
        for (int t = 0; t < ntile; ++t) {
          tc::mbar_arrive_expect_tx(b_full + 8 * t, p.b_tile_bytes);
          tc::bulk_load(smem_base + p.off_b + t * p.b_tile_bytes, wsrc + (size_t)t * p.b_tile_bytes, p.b_tile_bytes, b_full + 8 * t);
        }
    } else if (g == 0) {     // streamed weight tiles are shared by the groups of the CTA (same cout block, same plane range)
      RingPos b;
      for (int t = z_lo - p.Jhi; t <= z_end - 1 - p.Jlo; ++t) {
        if (t < 0 || t >= p.Din) continue;
        for (int c = 0; c < p.nclass; ++c) {
          if (max(t + p.cls[c].jlo, z_lo) > min(t + p.cls[c].jlo + p.cls[c].jcnt - 1, z_end - 1)) continue;
          const int ntaps = __popc(p.cls[c].tapmask);
          for (int kc = 0; kc < p.nkc; ++kc)
            for (int ti = 0; ti < ntaps; ++ti) {
              const int tile = kc * p.tiles_per_kc + p.cls[c].tile0 + ti;
              tc::mbar_wait(b_empty + 8 * b.idx, b.phase ^ 1, 2);
              if (leader) {
                tc::mbar_arrive_expect_tx(b_full + 8 * b.idx, p.b_tile_bytes);
                tc::bulk_load(smem_base + p.off_b + b.idx * p.b_tile_bytes, wsrc + (size_t)tile * p.b_tile_bytes, p.b_tile_bytes, b_full + 8 * b.idx);
              }
              b.advance(NB);
            }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer: warp-uniform control flow, one elected lane issues ---------------
    // A single warp has to sustain one tcgen05.mma per ~50 cycles on the narrow layers, so the code
    // between two MMAs is kept to a descriptor add: ring cursors instead of div/mod, and a straight-line
    // unrolled burst of 9 taps x KSTEPS per channel chunk in the steady state of a stride-1 layer.
    const bool elected = tc::elect_one();
    const bool leader = elected;
    if constexpr (FIRST && MULTI) {
      // one output plane per step: 6 MMAs per modality (weight tile m: 12 k8 chunks of CB rows), all into the plane's slot
      const uint32_t idesc = tc::instr_desc_f16(p.fmt, 128, (int)CB);
      const uint32_t hi_desc = (128u >> 4) | (1u << 14);
      const uint32_t a_lbo = (2048u >> 4) << 16, b_lbo = ((CB * 16u) >> 4) << 16;
      const uint32_t b_lo0 = (smem_b_d >> 4) | b_lbo;
      tc::mbar_wait(b_full, 0, 5);
      RingPos a, fresh, done;
      for (int t = z_lo; t < z_end; ++t) {
        tc::mbar_wait(acc_empty + 8 * fresh.idx, fresh.phase ^ 1, 3);
        const uint32_t col = tmem + fresh.idx * CB;
        for (int m = 0; m < NM; ++m) {
          tc::mbar_wait(a_mma + 8 * a.idx, a.phase, 4);
          tc::tc_fence_after();
          if (leader) {
            const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo;
            const uint32_t b_m = b_lo0 + (uint32_t)m * 12u * CB;
#pragma unroll
            for (int i = 0; i < 6; ++i) {
              const int achunk = (i == 0 || i == 4) ? 0 : (i == 1 || i == 5) ? 2 : (i == 2 ? 4 : 6);
              tc::umma_f16(col, tc_desc(hi_desc, a_lo0 + achunk * (2048 >> 4)), tc_desc(hi_desc, b_m + i * 2 * CB), idesc,
                           (m == 0 && i == 0) ? 0u : 1u);
            }
          }
          if (elected) tc::umma_commit(a_empty + 8 * a.idx);
          a.advance(SA);
          __syncwarp();
        }
        if (elected) tc::umma_commit(acc_full + 8 * done.idx);
        fresh.advance(R); done.advance(R);
        __syncwarp();
      }
    } else if constexpr (FIRST) {
      // one output plane per step: 6 MMAs (hi*w_hi, lo*w_hi, hi*w_lo; K = 32 each) into the plane's own slot
      const uint32_t idesc = tc::instr_desc_f16(p.fmt, 128, (int)CB);
      const uint32_t hi_desc = (128u >> 4) | (1u << 14);                  // SBO = 128 B for both operands
      const uint32_t a_lbo = (2048u >> 4) << 16, b_lbo = ((CB * 16u) >> 4) << 16;
      const uint32_t b_lo0 = (smem_b_d >> 4) | b_lbo;
      tc::mbar_wait(b_full, 0, 5);
      RingPos a, fresh, done;
      for (int t = z_lo; t < z_end; ++t) {
        tc::mbar_wait(acc_empty + 8 * fresh.idx, fresh.phase ^ 1, 3);
        tc::mbar_wait(a_mma + 8 * a.idx, a.phase, 4);
        tc::tc_fence_after();
        if (leader) {
          const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo;
          const uint32_t col = tmem + fresh.idx * CB;
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            const int achunk = (i == 0 || i == 4) ? 0 : (i == 1 || i == 5) ? 2 : (i == 2 ? 4 : 6);     // hi, hi, lo, lo, hi, hi
            tc::umma_f16(col, tc_desc(hi_desc, a_lo0 + achunk * (2048 >> 4)), tc_desc(hi_desc, b_lo0 + i * 2 * CB), idesc, i == 0 ? 0u : 1u);
          }
        }
        if (elected) { tc::umma_commit(a_empty + 8 * a.idx); tc::umma_commit(acc_full + 8 * done.idx); }
        a.advance(SA); fresh.advance(R); done.advance(R);
        __syncwarp();
      }
    } else {
    const uint32_t idesc0 = tc::instr_desc_f16(p.fmt, 128, 0);
    const uint32_t idesc1 = idesc0 | ((CB >> 3) << 17);
    const uint32_t b_lbo16 = (uint32_t)p.jmax * CB;                    // LBO of the weight tiles, in 16-B units
    const uint32_t kstep_b = 2u * b_lbo16, tile16 = p.b_tile_bytes >> 4;
    const uint32_t a_hi = (uint32_t)((TC_PW * 16) >> 4) | (1u << 14);  // SBO = 160 B, descriptor version 1
    const uint32_t b_hi = (128u >> 4) | (1u << 14);                    // SBO = 128 B
    const uint32_t a_lbo_field = (uint32_t)(TC_PLANE_BYTES >> 4) << 16;
    const uint32_t b_lo_res = (smem_b_d >> 4) | (b_lbo16 << 16);
    const int t_first = z_lo - p.Jhi, t_last_nominal = z_end - 1 - p.Jlo;
    const int last_t = min(t_last_nominal, p.Din - 1);
    const bool plain = p.nclass == 1 && p.Jlo == -1 && p.Jhi == 1;     // stride-1 3x3x3
    if (p.resident)
      for (int t = 0; t < p.nkc * p.tiles_per_kc; ++t) tc::mbar_wait(b_full + 8 * t, 0, 5);
    RingPos a, b, fresh, done;
    bool b_peek = false;      // same for the weight ring
    bool a_peek = false;      // a_full of the CURRENT stage already observed complete (prefetched try_wait)
    uint32_t lo_slot = 0;
    int next_fresh = z_lo, next_done = z_lo, zo_lo_prev = z_lo;
    for (int t = t_first; t <= t_last_nominal; ++t) {
      if (t < 0 || t >= p.Din) continue;
      const int zo_lo = max(t + p.Jlo, z_lo), zo_hi = min(t + p.Jhi, z_end - 1);
      if (zo_lo != zo_lo_prev) { lo_slot = (lo_slot + 1 == R) ? 0 : lo_slot + 1; zo_lo_prev = zo_lo; }
      const int fresh_from = next_fresh;        // output planes >= fresh_from are first touched in this step
      while (next_fresh <= zo_hi) {             // the epilogue must have drained the slot's previous use
        tc::mbar_wait(acc_empty + 8 * fresh.idx, fresh.phase ^ 1, 3);
        fresh.advance(R);
        ++next_fresh;
      }
      if (plain && zo_hi - zo_lo == 2 && R >= 3 && 3 * CB <= 256 && fresh_from == zo_hi) {
        // ---- steady state (interior plane, exactly output plane t+1 is new).  The three accumulator slots are
        // contiguous except at the ring wrap, where every MMA is issued as two (the general path is ~5x slower per MMA,
        // and 2 of every R planes straddle the wrap).  The issuer STAYS in this loop for the whole run of interior planes:
        // ncu's instruction-level samples showed it spending most of a plane in ~500 bookkeeping instructions of the outer
        // loop (constant-bank reloads of the kernel parameters, path selection) with the MMA queue full only a third of the time.
        const uint32_t id2 = idesc0 | (((2 * CB) >> 3) << 17), id3 = idesc0 | (((3 * CB) >> 3) << 17);
        // one copy of the loop per weight mode (resident / streamed): with both inline the loop body spanned 33 KB of SASS for
        // the ~240 instructions an iteration executes
        auto steady = [&](auto res_c) {
        constexpr bool RES = decltype(res_c)::value;
        for (;;) {
        const uint32_t col = tmem + lo_slot * CB;
        const bool wrap = lo_slot + 3 > R, wrapA = lo_slot + 2 == R;          // wrapA: slots R-2, R-1 | 0    else: R-1 | 0, 1
        const uint32_t idA = wrapA ? id2 : idesc1, idB = wrapA ? idesc1 : id2, offB = wrapA ? 2 * CB : CB;
        const uint32_t col1 = (lo_slot + 1 == R) ? tmem : col + CB, col2 = wrapA ? tmem : tmem + CB;      // slots lo+1, lo+2 when wrapping
        for (int kc = 0; kc < p.nkc; ++kc) {
          if (!a_peek) tc::mbar_wait(a_mma + 8 * a.idx, a.phase, 4);
          tc::tc_fence_after();
          { const RingPos an = a.next(SA); a_peek = tc::mbar_test_wait(a_mma + 8 * an.idx, an.phase); }   // result consumed after the burst
          if constexpr (!RES) {
            // streamed weight tiles: one ring slot per tap, shared by the groups of the CTA
            const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo_field;
#pragma unroll
            for (int sft = 0; sft < 9; ++sft) {
              if (!b_peek) tc::mbar_wait(b_full + 8 * b.idx, b.phase, 6);
              tc::tc_fence_after();
              const uint32_t b_lo0 = ((smem_b_d + b.idx * p.b_tile_bytes) >> 4) | (b_lbo16 << 16);
              { const RingPos bn = b.next(NB); b_peek = tc::mbar_test_wait(b_full + 8 * bn.idx, bn.phase); }
              if (leader) {
#pragma unroll
                for (int kk = 0; kk < KSTEPS; ++kk) {
                  const uint64_t adesc = tc_desc(a_hi, a_lo0 + (sft / 3) * TC_PW + (sft % 3) + kk * (2 * TC_PLANE_BYTES >> 4));
                  const uint32_t b0 = b_lo0 + kk * kstep_b;
                  const bool first = sft == 0 && kk == 0 && kc == 0;
                  if (!wrap) {
                    if (first) {
                      tc::umma_f16(col, adesc, tc_desc(b_hi, b0), id2, 1u);
                      tc::umma_f16(col + 2 * CB, adesc, tc_desc(b_hi, b0 + 2 * CB), idesc1, 0u);
                    } else tc::umma_f16(col, adesc, tc_desc(b_hi, b0), id3, 1u);
                  } else if (first) {
                    tc::umma_f16(col, adesc, tc_desc(b_hi, b0), idesc1, 1u);
                    tc::umma_f16(col1, adesc, tc_desc(b_hi, b0 + CB), idesc1, 1u);
                    tc::umma_f16(col2, adesc, tc_desc(b_hi, b0 + 2 * CB), idesc1, 0u);
                  } else {
                    tc::umma_f16(col, adesc, tc_desc(b_hi, b0), idA, 1u);
                    tc::umma_f16(tmem, adesc, tc_desc(b_hi, b0 + offB), idB, 1u);
                  }
                }
              }
              if (elected) tc::umma_commit(b_empty + 8 * b.idx);
              b.advance(NB);
            }
          } else if (leader && !wrap) {
            const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo_field;
            uint32_t bl = b_lo_res + (uint32_t)kc * 9u * tile16;
#pragma unroll
            for (int sft = 0; sft < 9; ++sft) {
#pragma unroll
              for (int kk = 0; kk < KSTEPS; ++kk) {
                const uint64_t adesc = tc_desc(a_hi, a_lo0 + (sft / 3) * TC_PW + (sft % 3) + kk * (2 * TC_PLANE_BYTES >> 4));
                if (sft == 0 && kk == 0) {
                  if (kc == 0) {     // first MMA of the plane: planes t-1, t accumulate, plane t+1 is overwritten
                    tc::umma_f16(col, adesc, tc_desc(b_hi, bl), id2, 1u);
                    tc::umma_f16(col + 2 * CB, adesc, tc_desc(b_hi, bl + 2 * CB), idesc1, 0u);
                  } else tc::umma_f16(col, adesc, tc_desc(b_hi, bl), id3, 1u);
                } else tc::umma_f16(col, adesc, tc_desc(b_hi, bl + kk * kstep_b), id3, 1u);
              }
              bl += tile16;
            }
          } else if (leader) {
            const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo_field;
            uint32_t bl = b_lo_res + (uint32_t)kc * 9u * tile16;
#pragma unroll
            for (int sft = 0; sft < 9; ++sft) {
#pragma unroll
              for (int kk = 0; kk < KSTEPS; ++kk) {
                const uint64_t adesc = tc_desc(a_hi, a_lo0 + (sft / 3) * TC_PW + (sft % 3) + kk * (2 * TC_PLANE_BYTES >> 4));
                const uint32_t b0 = bl + kk * kstep_b;
                if (sft == 0 && kk == 0 && kc == 0) {
                  tc::umma_f16(col, adesc, tc_desc(b_hi, b0), idesc1, 1u);
                  tc::umma_f16(col1, adesc, tc_desc(b_hi, b0 + CB), idesc1, 1u);
                  tc::umma_f16(col2, adesc, tc_desc(b_hi, b0 + 2 * CB), idesc1, 0u);
                } else {
                  tc::umma_f16(col, adesc, tc_desc(b_hi, b0), idA, 1u);
                  tc::umma_f16(tmem, adesc, tc_desc(b_hi, b0 + offB), idB, 1u);
                }
              }
              bl += tile16;
            }
          }
          if (elected) tc::umma_commit(a_empty + 8 * a.idx);
          a.advance(SA);
        }
        if (elected) tc::umma_commit(acc_full + 8 * done.idx);        // output plane t-1 is complete
        done.advance(R);
        ++next_done;
        __syncwarp();
        // is input plane t + 1 interior as well?  (its outputs t .. t + 2 inside the block, the plane itself inside the volume)
        if (t + 2 > z_end - 1 || t + 1 >= p.Din) break;
        ++t;
        lo_slot = (lo_slot + 1 == R) ? 0 : lo_slot + 1;           // the oldest live output plane is now t - 1
        zo_lo_prev = t - 1;
        tc::mbar_wait(acc_empty + 8 * fresh.idx, fresh.phase ^ 1, 3);      // output plane t + 1 starts
        fresh.advance(R);
        ++next_fresh;
        }
        };
        if (p.resident) steady(std::true_type{}); else steady(std::false_type{});
        continue;
      }
      if (p.nclass == 1 && p.Jlo == 0 && p.Jhi == 0 && p.tiles_per_kc == 9 && fresh_from == zo_hi) {
        // ---- 1x3x3 kernel, stride 1 (anisotropic plans): input plane t feeds output plane t alone -- 9 in-plane taps x
        // KSTEPS MMAs of N = CB per channel chunk into the plane's own slot; the first MMA overwrites it.
        const uint32_t col = tmem + lo_slot * CB;
        for (int kc = 0; kc < p.nkc; ++kc) {
          if (!a_peek) tc::mbar_wait(a_mma + 8 * a.idx, a.phase, 4);
          tc::tc_fence_after();
          { const RingPos an = a.next(SA); a_peek = tc::mbar_test_wait(a_mma + 8 * an.idx, an.phase); }
          const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo_field;
          uint32_t bl = b_lo_res + (uint32_t)kc * 9u * tile16;
#pragma unroll
          for (int sft = 0; sft < 9; ++sft) {
            uint32_t b_lo0 = bl;
            if (!p.resident) {
              if (!b_peek) tc::mbar_wait(b_full + 8 * b.idx, b.phase, 6);
              tc::tc_fence_after();
              b_lo0 = ((smem_b_d + b.idx * p.b_tile_bytes) >> 4) | (b_lbo16 << 16);
              { const RingPos bn = b.next(NB); b_peek = tc::mbar_test_wait(b_full + 8 * bn.idx, bn.phase); }
            }
            if (leader) {
#pragma unroll
              for (int kk = 0; kk < KSTEPS; ++kk) {
                const uint64_t adesc = tc_desc(a_hi, a_lo0 + (sft / 3) * TC_PW + (sft % 3) + kk * (2 * TC_PLANE_BYTES >> 4));
                tc::umma_f16(col, adesc, tc_desc(b_hi, b_lo0 + kk * kstep_b), idesc1, (sft == 0 && kk == 0 && kc == 0) ? 0u : 1u);
              }
            }
            if (!p.resident) {
              if (elected) tc::umma_commit(b_empty + 8 * b.idx);
              b.advance(NB);
            }
            bl += tile16;
          }
          if (elected) tc::umma_commit(a_empty + 8 * a.idx);
          a.advance(SA);
        }
        if (elected) tc::umma_commit(acc_full + 8 * done.idx);        // output plane t is complete
        done.advance(R);
        ++next_done;
        __syncwarp();
        continue;
      }
      if (p.s222 && zo_lo == t && zo_hi == t + 1 && fresh_from == zo_hi && 2 * CB <= 256) {
        // ---- steady state of a stride-(2,2,2) conv, straight line: the 8 parity classes and their 1/2/2/4 in-plane taps
        // are compile-time here (a tap LOOP costs more in loop / branch overhead than the two MMAs it issues -- tried twice:
        // the generic loop at ~250 cycles per tap, and a compact purpose-built loop that ran enc1-a at 1.90 instead of 1.67 ms).
        // Sub-plane t feeds output t (all classes) and t+1 (the four odd-depth classes, which come first: N = 2 CB); exactly
        // output t+1 is new.  One specialised copy per (weights resident?, ring wrap?) so that the copy that runs -- resident,
        // no wrap -- is contiguous code: with the four forms interleaved the ~900 instructions executed per plane were spread
        // over 48 KB of SASS and the issuer, the bottleneck of these layers, stalled on instruction fetch at every branch target.
        const uint32_t col0 = tmem + lo_slot * CB, col1 = (lo_slot + 1 == R) ? tmem : col0 + CB;
        const uint32_t id2 = idesc0 | (((2 * CB) >> 3) << 17);
        auto s222_step = [&](auto res_c, auto wrap_c) {
          constexpr bool RES = decltype(res_c)::value, WRAP = decltype(wrap_c)::value;
          uint32_t kstep = kstep_b;        // opaque: otherwise the offsets of all tiles x K steps are hoisted into the issuer's prologue and spill
          asm volatile("" : "+r"(kstep));
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const int cd = c >> 2, ph = (c >> 1) & 1, pw = c & 1;
            const int tile0 = cd * 9 + (ph ? (pw ? 5 : 3) : (pw ? 1 : 0));
            for (int kc = 0; kc < p.nkc; ++kc) {
              if (!a_peek) tc::mbar_wait(a_mma + 8 * a.idx, a.phase, 4);
              tc::tc_fence_after();
              { const RingPos an = a.next(SA); a_peek = tc::mbar_test_wait(a_mma + 8 * an.idx, an.phase); }
              const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo_field;
              const uint32_t b_res = b_lo_res + (uint32_t)(kc * p.tiles_per_kc + tile0) * tile16;
#pragma unroll
              for (int iy = 0; iy < (ph ? 2 : 1); ++iy) {
#pragma unroll
                for (int ix = 0; ix < (pw ? 2 : 1); ++ix) {
                  const int dy = ph ? iy : 1, dx = pw ? ix : 1, ti = iy * (pw ? 2 : 1) + ix;
                  uint32_t b_lo0;
                  if constexpr (RES) b_lo0 = b_res + ti * tile16;
                  else {
                    if (!b_peek) tc::mbar_wait(b_full + 8 * b.idx, b.phase, 6);
                    tc::tc_fence_after();
                    b_lo0 = ((smem_b_d + b.idx * p.b_tile_bytes) >> 4) | (b_lbo16 << 16);
                    { const RingPos bn = b.next(NB); b_peek = tc::mbar_test_wait(b_full + 8 * bn.idx, bn.phase); }
                  }
                  if (leader) {
#pragma unroll
                    for (int kk = 0; kk < KSTEPS; ++kk) {
                      const uint64_t adesc = tc_desc(a_hi, a_lo0 + dy * TC_PW + dx + kk * (2 * TC_PLANE_BYTES >> 4));
                      const uint32_t bl = b_lo0 + kk * kstep;
                      if (cd == 0) {
                        const bool first_site = c == 0 && kk == 0;             // the step's first MMA overwrites output t+1
                        if (WRAP || (first_site && kc == 0)) {
                          tc::umma_f16(col0, adesc, tc_desc(b_hi, bl), idesc1, 1u);
                          tc::umma_f16(col1, adesc, tc_desc(b_hi, bl + CB), idesc1, (first_site && kc == 0) ? 0u : 1u);
                        } else tc::umma_f16(col0, adesc, tc_desc(b_hi, bl), id2, 1u);
                      } else tc::umma_f16(col0, adesc, tc_desc(b_hi, bl), idesc1, 1u);
                    }
                  }
                  if constexpr (!RES) {
                    if (elected) tc::umma_commit(b_empty + 8 * b.idx);
                    b.advance(NB);
                  }
                }
              }
              if (elected) tc::umma_commit(a_empty + 8 * a.idx);
              a.advance(SA);
            }
          }
        };
        if (p.resident) { if (lo_slot + 1 == R) s222_step(std::true_type{}, std::true_type{}); else s222_step(std::true_type{}, std::false_type{}); }
        else { if (lo_slot + 1 == R) s222_step(std::false_type{}, std::true_type{}); else s222_step(std::false_type{}, std::false_type{}); }
        if (elected) tc::umma_commit(acc_full + 8 * done.idx);        // output plane t is complete
        done.advance(R);
        ++next_done;
        __syncwarp();
        continue;
      }
      if (p.Jlo == 0 && zo_lo == t && zo_hi == t + 1 && fresh_from == zo_hi && 2 * CB <= 256) {
        // ---- steady state of a depth-strided conv: sub-plane t feeds output t (all classes) and t+1 (odd-depth
        // classes, N = 2 CB); exactly output t+1 is new.  No segment bookkeeping, two MMAs only at the ring wrap.
        const uint32_t col0 = tmem + lo_slot * CB, col1 = (lo_slot + 1 == R) ? tmem : col0 + CB;
        const bool wrap = lo_slot + 1 == R;
        const uint32_t id2 = idesc0 | (((2 * CB) >> 3) << 17);
        bool fresh_pending = true;
        for (int c = 0; c < p.nclass; ++c) {
          const int jc = p.cls[c].jcnt, tapmask = p.cls[c].tapmask;
          for (int kc = 0; kc < p.nkc; ++kc) {
            if (!a_peek) tc::mbar_wait(a_mma + 8 * a.idx, a.phase, 4);
            tc::tc_fence_after();
            { const RingPos an = a.next(SA); a_peek = tc::mbar_test_wait(a_mma + 8 * an.idx, an.phase); }
            const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo_field;
            uint32_t b_res = b_lo_res + (uint32_t)(kc * p.tiles_per_kc + p.cls[c].tile0) * tile16;
            for (int m = tapmask; m; m &= m - 1) {
              const int sft = __ffs(m) - 1;
              uint32_t b_lo0;
              if (p.resident) { b_lo0 = b_res; b_res += tile16; }
              else {
                if (!b_peek) tc::mbar_wait(b_full + 8 * b.idx, b.phase, 6);
                tc::tc_fence_after();
                b_lo0 = ((smem_b_d + b.idx * p.b_tile_bytes) >> 4) | (b_lbo16 << 16);
                { const RingPos bn = b.next(NB); b_peek = tc::mbar_test_wait(b_full + 8 * bn.idx, bn.phase); }
              }
              const uint32_t a_lo1 = a_lo0 + (uint32_t)((kTapShift >> (5 * sft)) & 31u);
              if (leader) {
#pragma unroll
                for (int kk = 0; kk < KSTEPS; ++kk) {
                  const uint64_t adesc = tc_desc(a_hi, a_lo1 + kk * (2 * TC_PLANE_BYTES >> 4));
                  const uint32_t bl = b_lo0 + kk * kstep_b;
                  if (jc == 2) {
                    const bool fr = fresh_pending && kk == 0;
                    if (wrap || fr) {
                      tc::umma_f16(col0, adesc, tc_desc(b_hi, bl), idesc1, 1u);
                      tc::umma_f16(col1, adesc, tc_desc(b_hi, bl + CB), idesc1, fr ? 0u : 1u);
                    } else tc::umma_f16(col0, adesc, tc_desc(b_hi, bl), id2, 1u);
                  } else tc::umma_f16(col0, adesc, tc_desc(b_hi, bl), idesc1, 1u);
                }
              }
              if (jc == 2) fresh_pending = false;
              if (!p.resident) {
                if (elected) tc::umma_commit(b_empty + 8 * b.idx);
                b.advance(NB);
              }
            }
            if (elected) tc::umma_commit(a_empty + 8 * a.idx);
            a.advance(SA);
          }
        }
        if (elected) tc::umma_commit(acc_full + 8 * done.idx);        // output plane t is complete
        done.advance(R);
        ++next_done;
        __syncwarp();
        continue;
      }
      // ---- general path: parity classes, ring wrap, block edges, streamed weights -------------------
      bool first_mma = true;
      for (int c = 0; c < p.nclass; ++c) {
        const int dlo = max(t + p.cls[c].jlo, z_lo), dhi = min(t + p.cls[c].jlo + p.cls[c].jcnt - 1, z_end - 1);
        if (dlo > dhi) continue;
        const uint32_t cnt = (uint32_t)(dhi - dlo + 1), r0 = (uint32_t)(dlo - (t + p.cls[c].jlo));
        uint32_t sl = lo_slot + (uint32_t)(dlo - zo_lo);
        if (sl >= R) sl -= R;
        // column segments (split at the ring wrap and at N = 256), kept in scalars
        uint32_t nseg = 0, sc0 = 0, sc1 = 0, sc2 = 0, sb0 = 0, sb1 = 0, sb2 = 0, si0 = 0, si1 = 0, si2 = 0;
        {
          uint32_t i = 0;
          while (i < cnt) {
            const uint32_t slot = sl + i < R ? sl + i : sl + i - R;
            uint32_t len = min(cnt - i, R - slot);
            len = min(len, 256u / CB);
            const uint32_t c_ = tmem + slot * CB, b_ = (r0 + i) * CB, d_ = idesc0 | (((len * CB) >> 3) << 17);
            if (nseg == 0) { sc0 = c_; sb0 = b_; si0 = d_; } else if (nseg == 1) { sc1 = c_; sb1 = b_; si1 = d_; } else { sc2 = c_; sb2 = b_; si2 = d_; }
            ++nseg; i += len;
          }
        }
        const int tapmask = p.cls[c].tapmask;
        for (int kc = 0; kc < p.nkc; ++kc) {
          if (!a_peek) tc::mbar_wait(a_mma + 8 * a.idx, a.phase, 4);
          a_peek = false;
          tc::tc_fence_after();
          const uint32_t a_lo0 = ((smem_a_d + a.idx * p.a_stage_bytes) >> 4) | a_lbo_field;
          uint32_t b_res = b_lo_res + (uint32_t)(kc * p.tiles_per_kc + p.cls[c].tile0) * tile16;
          for (int m = tapmask; m; m &= m - 1) {
            const int sft = __ffs(m) - 1;
            uint32_t b_lo0;
            if (p.resident) { b_lo0 = b_res; b_res += tile16; }
            else {
              if (!b_peek) tc::mbar_wait(b_full + 8 * b.idx, b.phase, 6);
              tc::tc_fence_after();
              b_lo0 = ((smem_b_d + b.idx * p.b_tile_bytes) >> 4) | (b_lbo16 << 16);
              { const RingPos bn = b.next(NB); b_peek = tc::mbar_test_wait(b_full + 8 * bn.idx, bn.phase); }   // consumed at the next tap
            }
            const uint32_t a_lo1 = a_lo0 + (uint32_t)((kTapShift >> (5 * sft)) & 31u);
            if (first_mma) {
              // first MMA of the step: slot by slot, overwriting (accumulate = 0) first-touched slots
              for (uint32_t i = 0; i < cnt; ++i) {
                const uint32_t slot = sl + i < R ? sl + i : sl + i - R;
                if (leader) tc::umma_f16(tmem + slot * CB, tc_desc(a_hi, a_lo1), tc_desc(b_hi, b_lo0 + (r0 + i) * CB), idesc1,
                                         (dlo + (int)i) >= fresh_from ? 0u : 1u);
              }
            }
            if (leader) {
#pragma unroll
              for (int kk = 0; kk < KSTEPS; ++kk) {
                if (kk == 0 && first_mma) continue;
                const uint64_t adesc = tc_desc(a_hi, a_lo1 + kk * (2 * TC_PLANE_BYTES >> 4));
                const uint32_t bl = b_lo0 + kk * kstep_b;
                tc::umma_f16(sc0, adesc, tc_desc(b_hi, bl + sb0), si0, 1u);
                if (nseg > 1) tc::umma_f16(sc1, adesc, tc_desc(b_hi, bl + sb1), si1, 1u);
                if (nseg > 2) tc::umma_f16(sc2, adesc, tc_desc(b_hi, bl + sb2), si2, 1u);
              }
            }
            first_mma = false;
            if (!p.resident) {
              if (elected) tc::umma_commit(b_empty + 8 * b.idx);
              b.advance(NB);
            }
          }
          if (elected) tc::umma_commit(a_empty + 8 * a.idx);
          a.advance(SA);
        }
      }
      const int done_upto = (t == last_t) ? z_end - 1 : t + p.Jlo;
      while (next_done <= done_upto) {
        if (elected) tc::umma_commit(acc_full + 8 * done.idx);
        done.advance(R);
        ++next_done;
      }
      __syncwarp();
    }
    }   // !FIRST
  } else {
    // ---------------- epilogue: warps 2..5, TMEM lane quarter = warp % 4 ---------------------------
    const int q = warp_abs & 3;       // TMEM lane quarter is fixed by the hardware warp id
    const int row = q * 32 + lane;
    const int h = h0 + (row >> 3), w = w0 + (row & 7);
    const bool valid = h < p.H && w < p.W;
    const uint32_t tm_lane = tmem + ((uint32_t)(q * 32) << 16);
    const int nch = CB >> 4;
    if constexpr (TCONV) {
      // transposed conv (kernel == stride): column block q of the accumulator is output parity q; every
      // input voxel (GEMM row) scatters 16-byte channel chunks to its osd*osh*osw children.
      const int Ho = p.H * p.osh, Wo = p.W * p.osw;
      const size_t Vo = (size_t)p.D * p.osd * Ho * Wo;
      uint4* out_n = reinterpret_cast<uint4*>(p.out) + (size_t)n * (p.Cout_t >> 3) * Vo;
      uint32_t slot = 0, phase = 0;
      for (int t = z_lo; t < z_end; ++t) {
        tc::mbar_wait(acc_full + 8 * slot, phase, 7);
        tc::tc_fence_after();
        if (p.osw == 2) {
          // W-doubling (the usual case): the two W parities of a voxel are adjacent in memory, so a lane stores 32
          // contiguous bytes (full sectors, 256-bit stores) per 8-channel chunk instead of two half-sector writes.
          const int cpp = p.CBt >> 4;                              // 16-column chunks per parity block
          int chq = 0;                                             // first chunk of parity (qa, qb, qw = 0)
          for (int qa = 0; qa < p.osd; ++qa)
            for (int qb = 0; qb < p.osh; ++qb, chq += 2 * cpp)
              for (int cc = 0; cc < cpp; ++cc) {
                uint32_t r[2][16];
                tc::tmem_ld16(tm_lane + slot * CB + (chq + cc) * 16, r[0]);
                tc::tmem_ld16(tm_lane + slot * CB + (chq + cpp + cc) * 16, r[1]);
                tc::tmem_ld_wait();
                if (valid) {
                  float a0[16], a1[16];
#pragma unroll
                  for (int i = 0; i < 16; ++i) { a0[i] = __uint_as_float(r[0][i]); a1[i] = __uint_as_float(r[1][i]); }
                  uint4* o = out_n + (size_t)((cb * p.CBt + cc * 16) >> 3) * Vo + ((size_t)(t * p.osd + qa) * Ho + (h * p.osh + qb)) * Wo + (size_t)w * 2;
                  st_global_256(o, pack8<T>(a0), pack8<T>(a1));
                  st_global_256(o + Vo, pack8<T>(a0 + 8), pack8<T>(a1 + 8));
                }
              }
        } else {
        // two 16-column chunks per TMEM wait; the (parity, channel offset) of a chunk advances incrementally (no divisions)
        int cofs = 0, qa = 0, qb = 0, qw = 0;
        for (int ch = 0; ch < nch; ch += 2) {
          uint32_t r[2][16];
          tc::tmem_ld16(tm_lane + slot * CB + ch * 16, r[0]);
          tc::tmem_ld16(tm_lane + slot * CB + ch * 16 + 16, r[1]);
          tc::tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            float a[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) a[i] = __uint_as_float(r[u][i]);
            if (valid) {
              uint4* o = out_n + (size_t)((cb * p.CBt + cofs) >> 3) * Vo + ((size_t)(t * p.osd + qa) * Ho + (h * p.osh + qb)) * Wo + (w * p.osw + qw);
              o[0] = pack8<T>(a);
              o[Vo] = pack8<T>(a + 8);
            }
            cofs += 16;
            if (cofs == p.CBt) {
              cofs = 0;
              if (++qw == p.osw) { qw = 0; if (++qb == p.osh) { qb = 0; ++qa; } }
            }
          }
        }
        }
        tc::tc_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(acc_empty + 8 * slot);
        if (++slot == R) { slot = 0; phase ^= 1; }
      }
    } else {
    // InstanceNorm statistics (deterministic, no E[x^2] - E[x]^2 cancellation).  Every epilogue warp leaves one
    // (count, mean, M2) partial per channel in p.partials; stats_reduce_kernel combines them in a fixed order in fp64.
    //   SMALL_CB (CB <= 32): per-thread Welford recurrences for the thread's row over the planes (rs = mean, rq = M2), one
    //     transposing Chan reduction over the 32 rows at the end of the CTA;
    //   else: per plane a transposing shuffle reduction of (x - pivot), (x - pivot)^2 over the warp's 32 rows, the pivot
    //     being the running mean of the column (broadcast from its owner lane), merged into the lane's running (mean, M2).
    constexpr int NACC = SMALL_CB ? 32 : 8;
    float rs[NACC], rq[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i) { rs[i] = 0.f; rq[i] = 0.f; }
    float cnt = 0.f;                                                          // SMALL_CB: planes of this row; else: values per column so far
    const float nvw = (float)__popc(__ballot_sync(0xffffffffu, valid));       // valid rows of this warp
    const size_t V = (size_t)p.D * p.H * p.W;
    uint4* out_base = reinterpret_cast<uint4*>(p.out) + ((size_t)n * (p.Cout >> 3) + (size_t)cb * (CB >> 3)) * V;
    uint32_t slot = 0, phase = 0;
    for (int zo = z_lo; zo < z_end; ++zo) {
      tc::mbar_wait(acc_full + 8 * slot, phase, 7);
      tc::tc_fence_after();
      uint4* outp = out_base + ((size_t)zo * p.H + h) * p.W + w;
      float wgt_new, cnt_prev = cnt;
      if constexpr (SMALL_CB) { cnt += 1.f; wgt_new = __frcp_rn(cnt); }
      else { cnt += nvw; wgt_new = nvw > 0.f ? __fdividef(nvw, cnt) : 0.f; }
#pragma unroll
      for (int ch = 0; ch < (SMALL_CB ? 2 : 8); ++ch) {
        if (ch < nch) {
          uint32_t r[16];
          tc::tmem_ld16(tm_lane + slot * CB + ch * 16, r);
          tc::tmem_ld_wait();
          float a[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) a[i] = __uint_as_float(r[i]);
          if (valid) {
            if (p.out32) {
              float4* o32 = reinterpret_cast<float4*>(p.out) + 2 * (size_t)(outp - reinterpret_cast<uint4*>(p.out));
              o32[(size_t)(2 * ch) * V * 2] = make_float4(a[0], a[1], a[2], a[3]);
              o32[(size_t)(2 * ch) * V * 2 + 1] = make_float4(a[4], a[5], a[6], a[7]);
              o32[(size_t)(2 * ch + 1) * V * 2] = make_float4(a[8], a[9], a[10], a[11]);
              o32[(size_t)(2 * ch + 1) * V * 2 + 1] = make_float4(a[12], a[13], a[14], a[15]);
            } else {
              outp[(size_t)(2 * ch) * V] = pack8<T>(a);
              outp[(size_t)(2 * ch + 1) * V] = pack8<T>(a + 8);
            }
          }
          if constexpr (SMALL_CB) {
            if (valid) {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float d = a[i] - rs[ch * 16 + i];
                rs[ch * 16 + i] = fmaf(d, wgt_new, rs[ch * 16 + i]);
                rq[ch * 16 + i] = fmaf(d, a[i] - rs[ch * 16 + i], rq[ch * 16 + i]);
              }
            }
          } else {
            float b[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float piv = __shfl_sync(0xffffffffu, rs[ch], i);          // running mean of column i lives in lanes i, i + 16
              a[i] = valid ? a[i] - piv : 0.f;
              b[i] = a[i] * a[i];
            }
            // transposing butterfly: afterwards lane l holds the 32-row total of column (l & 15)
#pragma unroll
            for (int k = 8; k >= 1; k >>= 1) {
              const bool up = (lane & k) != 0;
#pragma unroll
              for (int i = 0; i < k; ++i) {
                const float sa_ = up ? a[i] : a[i + k], ka_ = up ? a[i + k] : a[i];
                const float sb_ = up ? b[i] : b[i + k], kb_ = up ? b[i + k] : b[i];
                a[i] = ka_ + __shfl_xor_sync(0xffffffffu, sa_, k);
                b[i] = kb_ + __shfl_xor_sync(0xffffffffu, sb_, k);
              }
            }
            const float S = a[0] + __shfl_xor_sync(0xffffffffu, a[0], 16), Q = b[0] + __shfl_xor_sync(0xffffffffu, b[0], 16);
            if (nvw > 0.f) {
              // this plane's block: nvw values, mean = pivot + S / nvw, M2 = Q - S^2 / nvw; the pivot IS the running mean
              const float dm = S / nvw;
              rq[ch] += fmaf(-S, dm, Q) + dm * dm * cnt_prev * wgt_new;
              rs[ch] = fmaf(dm, wgt_new, rs[ch]);
            }
          }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(acc_empty + 8 * slot);
      if (++slot == R) { slot = 0; phase ^= 1; }
    }
    // the four epilogue warps park their partials in this group's (now idle) activation ring: every MMA that read it and
    // every copy that wrote it completed before the last acc_full; combined after the CTA-wide barrier below
    StatPartial* pout = reinterpret_cast<StatPartial*>(smem + (size_t)g * SA * p.a_stage_bytes) + (size_t)q * CB;
    if constexpr (SMALL_CB) {
      // one transposing reduction for the whole CTA lifetime: Chan's merge of the rows' (count, mean, M2)
      const float n_row = valid ? cnt : 0.f;
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        if (ch < nch) {
          float a[16], b[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) { a[i] = rs[ch * 16 + i]; b[i] = rq[ch * 16 + i]; }
          float nn = n_row;
#pragma unroll
          for (int k = 8; k >= 1; k >>= 1) {
            const bool up = (lane & k) != 0;
            const float np_ = __shfl_xor_sync(0xffffffffu, nn, k);
            const float nt = nn + np_, wp = nt > 0.f ? np_ / nt : 0.f;
#pragma unroll
            for (int i = 0; i < k; ++i) {
              const float sa_ = up ? a[i] : a[i + k], ka_ = up ? a[i + k] : a[i];
              const float sb_ = up ? b[i] : b[i + k], kb_ = up ? b[i + k] : b[i];
              const float pm = __shfl_xor_sync(0xffffffffu, sa_, k), pq = __shfl_xor_sync(0xffffffffu, sb_, k);
              const float d = pm - ka_;
              a[i] = fmaf(d, wp, ka_);
              b[i] = kb_ + pq + d * d * nn * wp;
            }
            nn = nt;
          }
          // lanes l and l ^ 16 hold the two halves of column (l & 15): the lower lane merges and stores
          const float np_ = __shfl_xor_sync(0xffffffffu, nn, 16), pm = __shfl_xor_sync(0xffffffffu, a[0], 16), pq = __shfl_xor_sync(0xffffffffu, b[0], 16);
          float m_ = a[0], q_ = b[0];
          stat_merge<float>(nn, m_, q_, np_, pm, pq);
          if (lane < 16) *reinterpret_cast<float4*>(pout + ch * 16 + lane) = make_float4(nn, m_, q_, 0.f);
        }
      }
    } else if (lane < 16) {
#pragma unroll
      for (int ch = 0; ch < 8; ++ch)
        if (ch < nch) *reinterpret_cast<float4*>(pout + ch * 16 + lane) = make_float4(cnt, rs[ch], rq[ch], 0.f);
    }
    }   // !TCONV
  }
  tc::tc_fence_before();
  __syncthreads();
  if constexpr (!TCONV) {
    // one (count, mean, M2) partial per work item and channel: the four warps' partials merged in warp order
    for (int i = threadIdx.x; i < p.G * (int)CB; i += blockDim.x) {
      const int gg = i / (int)CB, c_ = i - gg * (int)CB;
      if ((int)blockIdx.x * p.G + gg >= p.total_items) continue;          // idle second group of the last CTA
      const StatPartial* pin = reinterpret_cast<const StatPartial*>(smem + (size_t)gg * SA * p.a_stage_bytes) + c_;
      float4 v = *reinterpret_cast<const float4*>(pin);
#pragma unroll
      for (int qq = 1; qq < 4; ++qq) {
        const float4 u = *reinterpret_cast<const float4*>(pin + (size_t)qq * CB);
        stat_merge<float>(v.x, v.y, v.z, u.x, u.y, u.z);
      }
      *reinterpret_cast<float4*>(p.partials + (size_t)(blockIdx.x * p.G + gg) * CB + c_) = v;
    }
  }
  if (warp_abs == 1) tc::tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------
// host side: configuration, weight packing, tensor maps, launch
// ------------------------------------------------------------------------------------------------
struct TcLayer {
  bool enabled = false;
  int ms0[6] = {0, 0, 0, 0, 0, 0}, ms1[6] = {0, 0, 0, 0, 0, 0};   // tensor-map specs {n, C, D, H, W, KC}; ms1[0] == 0 -> no second input
  bool map_bf16 = false;
  bool xform_ok = false;          // layer shape supports norm-on-load of its (single) input: plain stride-1, 32-channel chunks, resident weights
  CUtensorMap tm0, tm1;
  void* wpack = nullptr;
  TcKParams kp{};
  size_t smem_bytes = 0;
};

inline void tc_free(TcLayer& t) {
  if (t.wpack) cudaFree(t.wpack);
  t.wpack = nullptr;
  t.enabled = false;
}

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_tmapEncodeTiled tc_encode_fn() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(f);
  }
  return fn;
}

// tensor map over one activation tensor [maxN][C/8][D][H][W][8]: dims (W*8, H, D, maxN*C/8), box (80, 18, 1, KC/8)
inline bool tc_make_map(CUtensorMap* m, const void* base, int maxN, int C, int D, int H, int W, int KC, bool bf16, std::string* why) {
  PFN_tmapEncodeTiled enc = tc_encode_fn();
  if (!enc) { *why = "cuTensorMapEncodeTiled unavailable"; return false; }
  cuuint64_t dims[4] = {(cuuint64_t)W * 8, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)maxN * (C / 8)};
  cuuint64_t strides[3] = {(cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)D * H * W * 16};
  cuuint32_t box[4] = {TC_PW * 8, TC_PH, 1, (cuuint32_t)(KC / 8)};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { *why = "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r); return false; }
  return true;
}

// (re)encode the input tensor maps of a prepared layer for another set of activation buffers
inline int tc_remap(TcLayer& t, const void* in0, const void* in1, std::string* why) {
  if (!tc_make_map(&t.tm0, in0, t.ms0[0], t.ms0[1], t.ms0[2], t.ms0[3], t.ms0[4], t.ms0[5], t.map_bf16, why)) return 1;
  if (t.ms1[0] > 0) { if (!tc_make_map(&t.tm1, in1, t.ms1[0], t.ms1[1], t.ms1[2], t.ms1[3], t.ms1[4], t.ms1[5], t.map_bf16, why)) return 1; }
  else t.tm1 = t.tm0;
  return 0;
}

inline uint16_t tc_to_bits(float v, bool bf16) {
  if (bf16) { __nv_bfloat16 h = __float2bfloat16_rn(v); return *reinterpret_cast<uint16_t*>(&h); }
  __half h = __float2half_rn(v);
  return *reinterpret_cast<uint16_t*>(&h);
}

// Class order index of a voxel parity in the parity-split copy (must match tc_prepare's class loop:
// odd D-parity first, so the first class of a step touches every freshly started output plane).
__host__ __device__ inline int tc_s2d_class(int d, int h, int w, int sd, int sh, int sw) {
  const int cd = sd == 2 ? 1 - (d & 1) : 0, ch = sh == 2 ? (h & 1) : 0, cw = sw == 2 ? (w & 1) : 0;
  return (cd * sh + ch) * sw + cw;
}

// Returns 0 always; t.enabled says whether the layer runs on the tensor cores.  *why is set only on
// a hard failure of a layer that should have been supported.  For a strided layer `in0` must be the
// parity-split copy of the producer tensor.
inline int tc_prepare(TcLayer& t, const std::vector<float>& w, int c0, int c1, int cout, const int k[3], const int s[3],
                      const int in_sp[3], const int out_sp[3], int maxN, bool bf16, const void* in0, const void* in1,
                      void* out, bool out32, std::string* why) {
  t.enabled = false;
  why->clear();
  // 3x3x3, or 1x3x3 (anisotropic plans: no taps and no stride along the thick-slice axis, SURVEY A8)
  if ((k[0] != 3 && k[0] != 1) || k[1] != 3 || k[2] != 3) return 0;
  const int kd = k[0];
  if (kd == 1 && s[0] != 1) return 0;
  const bool strided = s[0] != 1 || s[1] != 1 || s[2] != 1;
  if (strided && c1 > 0) return 0;
  if (c0 % 16 || c1 % 16 || cout % 16) return 0;
  const int cin = c0 + c1;
  TcKParams& kp = t.kp;
  // ---- parity classes ----
  const int sd = s[0], sh = s[1], sw = s[2];
  kp.out32 = out32 ? 1 : 0;
  kp.tconv = 0; kp.CBt = 0; kp.osd = kp.osh = kp.osw = 1; kp.Cout_t = cout;
  kp.nclass = sd * sh * sw; kp.Jlo = (sd == 1 && kd == 3) ? -1 : 0; kp.Jhi = kd == 3 ? 1 : 0; kp.jmax = kd == 1 ? 1 : (sd == 1 ? 3 : 2);
  kp.Din = in_sp[0] / sd;
  struct Tap { int kh, kw; };
  std::vector<std::vector<Tap>> cls_taps(kp.nclass);
  std::vector<std::vector<int>> cls_kd(kp.nclass);
  int tile0 = 0;
  for (int cd = 0; cd < sd; ++cd)
    for (int ph = 0; ph < sh; ++ph)
      for (int pw = 0; pw < sw; ++pw) {
        const int c = (cd * sh + ph) * sw + pw;
        const int pd = sd == 2 ? 1 - cd : 0;
        TcClassDesc& cd_ = kp.cls[c];
        cd_.tapmask = 0; cd_.tile0 = tile0;
        if (kd == 1) { cd_.jlo = 0; cd_.jcnt = 1; cls_kd[c] = {0}; }
        else if (sd == 1) { cd_.jlo = -1; cd_.jcnt = 3; cls_kd[c] = {2, 1, 0}; }
        else if (pd == 0) { cd_.jlo = 0; cd_.jcnt = 1; cls_kd[c] = {1}; }
        else { cd_.jlo = 0; cd_.jcnt = 2; cls_kd[c] = {2, 0}; }
        for (int dy = 0; dy < 3; ++dy)
          for (int dx = 0; dx < 3; ++dx) {
            int kh = -1, kw = -1;
            if (sh == 1) kh = dy; else if (ph == 0) { if (dy == 1) kh = 1; } else { if (dy == 0) kh = 0; else if (dy == 1) kh = 2; }
            if (sw == 1) kw = dx; else if (pw == 0) { if (dx == 1) kw = 1; } else { if (dx == 0) kw = 0; else if (dx == 1) kw = 2; }
            if (kh < 0 || kw < 0) continue;
            cd_.tapmask |= 1 << (dy * 3 + dx);
            cls_taps[c].push_back({kh, kw});
          }
        tile0 += (int)cls_taps[c].size();
      }
  kp.tiles_per_kc = tile0;
  // the straight-line stride-(2,2,2) issue path hard-codes this table: verify it instead of assuming it
  kp.s222 = (sd == 2 && sh == 2 && sw == 2 && kp.nclass == 8 && tile0 == 18) ? 1 : 0;
  for (int c = 0; c < 8 && kp.s222; ++c) {
    const int cd = c >> 2, ph = (c >> 1) & 1, pw = c & 1;
    int mask = 0;
    for (int iy = 0; iy < (ph ? 2 : 1); ++iy)
      for (int ix = 0; ix < (pw ? 2 : 1); ++ix) mask |= 1 << ((ph ? iy : 1) * 3 + (pw ? ix : 1));
    const TcClassDesc& d = kp.cls[c];
    if (d.tapmask != mask || d.tile0 != cd * 9 + (ph ? (pw ? 5 : 3) : (pw ? 1 : 0)) || d.jlo != 0 || d.jcnt != (cd == 0 ? 2 : 1)) kp.s222 = 0;
  }
  // ---- tiling / shared-memory plan ----
  int KC0 = 64;
  while (KC0 > 16 && (c0 % KC0 || c1 % KC0)) KC0 >>= 1;
  const int budget = TC_SMEM_MAX - TC_SMEM_RESERVED;
  int KC = 0, CB = 0, SA = 0, NB = 0, resident = 0, G = 1;
  // (1) dual-group resident plan: two tile pipelines share the resident weights (each gets 256 TMEM columns)
  for (int kc = KC0; kc >= 16 && !CB; kc >>= 1) {
    const int a_stage = kc * 360, ntile = (cin / kc) * kp.tiles_per_kc;
    if (ntile > TC_MAX_NB) continue;
    for (int cbt = std::min(cout, 64); cbt >= 32; cbt -= 16) {
      if (cout % cbt) continue;
      const long long btot = (long long)ntile * kp.jmax * cbt * kc * 2;
      if (btot + 2LL * 3 * a_stage <= budget) {
        KC = kc; CB = cbt; resident = 1; NB = ntile; G = 2;
        SA = (int)std::min<long long>(TC_MAX_SA, (budget - btot) / (2LL * a_stage));
        break;
      }
    }
  }
  // (1b) dual-group streaming plan: both groups consume ONE shared ring of weight tiles in lockstep (M = 256 per tile fetched)
  for (int kc = KC0; kc >= 32 && !CB; kc >>= 1) {
    const int a_stage = kc * 360;
    for (int cbt = std::min(cout, 64); cbt >= 32; cbt -= 16) {
      if (cout % cbt) continue;
      if (256 / cbt < kp.jmax + 1) continue;
      const int b_tile = kp.jmax * cbt * kc * 2;
      const int nb = (budget - 2 * 3 * a_stage) / b_tile;
      if (nb >= 3) { KC = kc; CB = cbt; resident = 0; SA = 3; NB = std::min(nb, TC_MAX_NB); G = 2; break; }
    }
  }
  // (2) single-group plans
  for (int kc = KC0; kc >= 16 && !CB; kc >>= 1) {
    const int a_stage = kc * 360, ntile = (cin / kc) * kp.tiles_per_kc;
    if (ntile <= TC_MAX_NB) {
      for (int cbt = std::min(cout, 128); cbt >= 16; cbt -= 16) {
        if (cout % cbt) continue;
        if (cbt < 32 && cbt != cout) break;
        const long long btot = (long long)ntile * kp.jmax * cbt * kc * 2;
        if (btot + 2LL * a_stage <= budget) {
          KC = kc; CB = cbt; resident = 1; NB = ntile;
          SA = (int)std::min<long long>(TC_MAX_SA, (budget - btot) / a_stage);
          break;
        }
      }
    }
    if (!CB) {      // streaming weights
      for (int cbt = std::min(cout, 128); cbt >= 16; cbt -= 16) {
        if (cout % cbt) continue;
        const int b_tile = kp.jmax * cbt * kc * 2;
        const int nb = (budget - 3 * a_stage) / b_tile;
        if (nb >= 3) { KC = kc; CB = cbt; resident = 0; SA = 3; NB = std::min(nb, TC_MAX_NB); break; }
      }
    }
  }
  if (!CB) return 0;
  kp.C0 = c0; kp.C1 = c1; kp.Cout = cout; kp.CB = CB; kp.KC = KC; kp.nkc = cin / KC; kp.nkc0 = c0 / KC;
  kp.D = out_sp[0]; kp.H = out_sp[1]; kp.W = out_sp[2];
  kp.tilesH = (kp.H + TC_TH - 1) / TC_TH; kp.tilesW = (kp.W + TC_TW - 1) / TC_TW;
  kp.ncb = cout / CB; kp.SA = SA; kp.NB = NB; kp.resident = resident; kp.G = G;
  kp.xf_src = nullptr;
  kp.xform = 0; kp.xf_sums = nullptr; kp.xf_gamma = nullptr; kp.xf_beta = nullptr; kp.xf_inv_count = 0.0;
  t.xform_ok = !strided && kd == 3 && resident && c1 == 0 && KC == 32 && (cin == 32 || cin == 64) && CB <= 32 && SA >= 3;
  kp.R = std::min(TC_MAX_R, (512 / G) / CB);
  kp.fmt = bf16 ? 1 : 0;
  kp.a_stage_bytes = KC * 360; kp.b_tile_bytes = kp.jmax * CB * KC * 2;
  kp.off_b = G * SA * kp.a_stage_bytes;
  kp.off_bar = kp.off_b + NB * kp.b_tile_bytes;
  kp.off_bar = (kp.off_bar + 127) & ~127u;
  t.smem_bytes = kp.off_bar + TC_SMEM_RESERVED;
  if (t.smem_bytes > TC_SMEM_MAX) { *why = "internal: shared memory plan exceeds 227 KB"; return 1; }
  if (t.smem_bytes < 120 * 1024) t.smem_bytes = 120 * 1024;          // one CTA per SM: the CTA owns all 512 TMEM columns
  kp.out = out;
  // ---- operand tiles: [cb][kc][class, tap][k8][row = r*CB + co][8]; row block r <-> output plane t+jlo+r ----
  const size_t tile_elems = (size_t)(KC / 8) * kp.jmax * CB * 8;
  const int ntile = kp.nkc * kp.tiles_per_kc;
  std::vector<uint16_t> pk((size_t)kp.ncb * ntile * tile_elems, 0);
  for (int cb = 0; cb < kp.ncb; ++cb)
    for (int kc = 0; kc < kp.nkc; ++kc)
      for (int c = 0; c < kp.nclass; ++c)
        for (size_t ti = 0; ti < cls_taps[c].size(); ++ti) {
          uint16_t* tile = pk.data() + ((size_t)cb * ntile + (size_t)kc * kp.tiles_per_kc + kp.cls[c].tile0 + ti) * tile_elems;
          for (int k8 = 0; k8 < KC / 8; ++k8)
            for (int r = 0; r < kp.cls[c].jcnt; ++r)
              for (int co_ = 0; co_ < CB; ++co_)
                for (int e = 0; e < 8; ++e) {
                  const int co = cb * CB + co_, ci = kc * KC + k8 * 8 + e;
                  const float v = w[((size_t)co * cin + ci) * (kd * 9) + cls_kd[c][r] * 9 + cls_taps[c][ti].kh * 3 + cls_taps[c][ti].kw];
                  tile[((size_t)k8 * kp.jmax * CB + (size_t)r * CB + co_) * 8 + e] = tc_to_bits(v, bf16);
                }
        }
  if (cudaMalloc(&t.wpack, pk.size() * 2) != cudaSuccess) { *why = "cudaMalloc(wpack) failed"; return 1; }
  if (cudaMemcpy(t.wpack, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) { *why = "cudaMemcpy(wpack) failed"; return 1; }
  kp.wpack = t.wpack;
  // input maps: the (possibly parity-split) producer tensor has nclass * C0 channels at the reduced resolution
  t.map_bf16 = bf16;
  { const int a0[6] = {maxN * kp.nclass, c0, in_sp[0] / sd, in_sp[1] / sh, in_sp[2] / sw, KC}; for (int i = 0; i < 6; ++i) t.ms0[i] = a0[i]; }
  { const int a1[6] = {c1 > 0 ? maxN : 0, c1, in_sp[0], in_sp[1], in_sp[2], KC}; for (int i = 0; i < 6; ++i) t.ms1[i] = a1[i]; }
  if (tc_remap(t, in0, in1, why)) return 1;
  t.enabled = true;
  return 0;
}

// Transposed conv with kernel == stride (1 or 2 per axis), no bias: a 1-tap GEMM over the INPUT voxels whose
// N dimension stacks the osd*osh*osw output parities; w in PyTorch layout [Cin][Cout][kd][kh][kw].
inline int tc_prepare_tconv(TcLayer& t, const std::vector<float>& w, int cin, int cout, const int s[3], const int in_sp[3],
                            int maxN, bool bf16, const void* in0, void* out, std::string* why) {
  t.enabled = false;
  why->clear();
  if (cin % 16 || cout % 16) return 0;
  const int nco = s[0] * s[1] * s[2];
  int CBt = 256 / nco;
  while (CBt >= 16 && (cout % CBt || CBt % 16)) CBt -= 16;
  if (CBt < 16) return 0;
  TcKParams& kp = t.kp;
  kp = TcKParams{};
  kp.tconv = 1; kp.CBt = CBt; kp.osd = s[0]; kp.osh = s[1]; kp.osw = s[2]; kp.Cout_t = cout;
  kp.nclass = 1; kp.Jlo = 0; kp.Jhi = 0; kp.jmax = 1; kp.tiles_per_kc = 1; kp.Din = in_sp[0];
  kp.cls[0] = TcClassDesc{1 << 4, 0, 1, 0};
  const int CB = nco * CBt;
  if (CB % 32) return 0;                 // the scatter epilogue reads two 16-column chunks per step
  int KC = 64;
  while (KC > 16 && cin % KC) KC >>= 1;
  const int budget = TC_SMEM_MAX - TC_SMEM_RESERVED;
  const int a_stage = KC * 360, b_tile = CB * KC * 2, nkc = cin / KC;
  int SA, NB, resident;
  if (nkc <= TC_MAX_NB && (long long)nkc * b_tile + 2LL * a_stage <= budget) {
    resident = 1; NB = nkc; SA = (int)std::min<long long>(TC_MAX_SA, (budget - (long long)nkc * b_tile) / a_stage);
  } else {
    resident = 0; SA = 3; NB = std::min((budget - 3 * a_stage) / b_tile, TC_MAX_NB);
    if (NB < 2) return 0;
  }
  kp.C0 = cin; kp.C1 = 0; kp.Cout = CB * (cout / CBt); kp.CB = CB; kp.KC = KC; kp.nkc = nkc; kp.nkc0 = nkc;
  kp.D = in_sp[0]; kp.H = in_sp[1]; kp.W = in_sp[2];
  kp.tilesH = (kp.H + TC_TH - 1) / TC_TH; kp.tilesW = (kp.W + TC_TW - 1) / TC_TW;
  kp.ncb = cout / CBt; kp.SA = SA; kp.NB = NB; kp.resident = resident;
  kp.R = 512 / CB; kp.fmt = bf16 ? 1 : 0; kp.G = 1;
  kp.a_stage_bytes = a_stage; kp.b_tile_bytes = b_tile;
  kp.off_b = SA * a_stage;
  kp.off_bar = (kp.off_b + NB * b_tile + 127) & ~127u;
  t.smem_bytes = kp.off_bar + TC_SMEM_RESERVED;
  if (t.smem_bytes > TC_SMEM_MAX) { *why = "internal: shared memory plan exceeds 227 KB"; return 1; }
  if (t.smem_bytes < 120 * 1024) t.smem_bytes = 120 * 1024;
  kp.out = out;
  const int taps = nco;
  const size_t tile_elems = (size_t)(KC / 8) * CB * 8;
  std::vector<uint16_t> pk((size_t)kp.ncb * nkc * tile_elems, 0);
  for (int cb = 0; cb < kp.ncb; ++cb)
    for (int kc = 0; kc < nkc; ++kc) {
      uint16_t* tile = pk.data() + ((size_t)cb * nkc + kc) * tile_elems;
      for (int k8 = 0; k8 < KC / 8; ++k8)
        for (int q = 0; q < nco; ++q)
          for (int co_ = 0; co_ < CBt; ++co_)
            for (int e = 0; e < 8; ++e) {
              const int ci = kc * KC + k8 * 8 + e, co = cb * CBt + co_;
              tile[((size_t)k8 * CB + (size_t)q * CBt + co_) * 8 + e] = tc_to_bits(w[((size_t)ci * cout + co) * taps + q], bf16);
            }
    }
  if (cudaMalloc(&t.wpack, pk.size() * 2) != cudaSuccess) { *why = "cudaMalloc(wpack) failed"; return 1; }
  if (cudaMemcpy(t.wpack, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) { *why = "cudaMemcpy(wpack) failed"; return 1; }
  kp.wpack = t.wpack;
  t.map_bf16 = bf16;
  { const int a0[6] = {maxN, cin, in_sp[0], in_sp[1], in_sp[2], KC}; for (int i = 0; i < 6; ++i) t.ms0[i] = a0[i]; }
  t.ms1[0] = 0;
  if (tc_remap(t, in0, nullptr, why)) return 1;
  t.enabled = true;
  return 0;
}

// First conv (Cin = 1, 3x3x3, stride 1): the loader warps of the FIRST kernel build the [128 voxels][32 taps] im2col
// operand of every output plane from the fp32 volume (tile origin + mirror flip applied on the fly); input and weights
// are split hi + lo into two fp16 (bf16) values, so the 6 MMAs per plane (hi*w_hi, lo*w_hi, hi*w_lo) reproduce the fp32
// product to ~2^-22.  w27 = weights as [modality][tap][Cout] (tap = (kd*3 + kh)*3 + kw).
// nmod > 1 (MULTI kernel): one stage and one 12-chunk weight tile per modality, a 4 * nmod-slot slice ring per group.
inline int tc_prepare_first(TcLayer& t, const std::vector<float>& w27, int cout, const int sp[3], bool bf16, void* out, std::string* why,
                            int nmod = 1) {
  t.enabled = false;
  why->clear();
  if (cout != 16 && cout != 32) return 0;
  if (nmod < 1 || nmod > 4) return 0;
  TcKParams& kp = t.kp;
  kp = TcKParams{};
  kp.first = 1;
  kp.nclass = 1; kp.Jlo = 0; kp.Jhi = 0; kp.jmax = 1; kp.tiles_per_kc = 1; kp.Din = sp[0];
  kp.cls[0] = TcClassDesc{1 << 4, 0, 1, 0};
  kp.C0 = 8; kp.C1 = 0; kp.Cout = cout; kp.CB = cout; kp.KC = 32; kp.nkc = 1; kp.nkc0 = 1;
  kp.D = sp[0]; kp.H = sp[1]; kp.W = sp[2];
  kp.tilesH = (kp.H + TC_TH - 1) / TC_TH; kp.tilesW = (kp.W + TC_TW - 1) / TC_TW;
  kp.ncb = 1; kp.SA = TC_MAX_SA; kp.NB = 1; kp.resident = 1;
  kp.R = std::min(TC_MAX_R, 256 / cout); kp.fmt = bf16 ? 1 : 0; kp.G = 2;
  kp.a_stage_bytes = TC_FIRST_STAGE_BYTES; kp.b_tile_bytes = 12 * cout * 16 * nmod;
  kp.off_b = kp.G * kp.SA * kp.a_stage_bytes;
  kp.off_bar = (kp.off_b + kp.b_tile_bytes + 127) & ~127u;
  if (nmod == 1) t.smem_bytes = kp.off_bar + TC_SMEM_RESERVED_FIRST;
  else {
    // after off_bar (the kernel's layout): G * nbar barriers, TMEM pointer, coefficient area, G * 4 * nmod slices, slice barriers
    const uint32_t nbar = 3 * kp.SA + 2 * kp.NB + 2 * kp.R;
    const uint32_t aux = (8u * nbar * kp.G + 24u) & ~15u;
    const uint32_t slices_end = aux + 4u * (kp.G * 2 * kp.CB + kp.G * 2 * 64 + kp.G * 4 * nmod * TC_FIRST_SLICE);
    kp.fc_sbar = (slices_end + 7u) & ~7u;
    kp.fc_M = nmod;
    t.smem_bytes = kp.off_bar + kp.fc_sbar + kp.G * 256;
  }
  if (t.smem_bytes > TC_SMEM_MAX) { *why = "internal: shared memory plan exceeds 227 KB"; return 1; }
  kp.out = out;
  // B tile of modality m: [12 k8 chunks][cout rows][8]: K blocks of 16 taps = w_hi(0-15), w_hi(16-31), w_hi(0-15), w_hi(16-31),
  // w_lo(0-15), w_lo(16-31)
  auto from_bits = [&](uint16_t b) -> float {
    if (bf16) { uint32_t u = (uint32_t)b << 16; float f; memcpy(&f, &u, 4); return f; }
    __half h; memcpy(&h, &b, 2); return __half2float(h);
  };
  std::vector<uint16_t> pk((size_t)nmod * 12 * cout * 8, 0);
  for (int m = 0; m < nmod; ++m)
  for (int kb = 0; kb < 6; ++kb)
    for (int k8 = 0; k8 < 2; ++k8)
      for (int co = 0; co < cout; ++co)
        for (int e = 0; e < 8; ++e) {
          const int tap = (kb & 1) * 16 + k8 * 8 + e;
          uint16_t v = 0;
          if (tap < 27) {
            const float wf = w27[((size_t)m * 27 + tap) * cout + co];
            const uint16_t hi = tc_to_bits(wf, bf16);
            v = kb < 4 ? hi : tc_to_bits(wf - from_bits(hi), bf16);
          }
          pk[(((size_t)m * 12 + kb * 2 + k8) * cout + co) * 8 + e] = v;
        }
  if (cudaMalloc(&t.wpack, pk.size() * 2) != cudaSuccess) { *why = "cudaMalloc(wpack) failed"; return 1; }
  if (cudaMemcpy(t.wpack, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) { *why = "cudaMemcpy(wpack) failed"; return 1; }
  kp.wpack = t.wpack;
  t.map_bf16 = bf16;
  t.ms0[0] = 0; t.ms1[0] = 0;
  memset(&t.tm0, 0, sizeof t.tm0); memset(&t.tm1, 0, sizeof t.tm1);
  t.enabled = true;
  return 0;
}

template <typename T>
inline int tc_set_attr_all() {
  cudaError_t e = cudaSuccess;
#define DWMH_TC_ATTR(K, S, C, D) if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3_tc_kernel<T, K, S, C, D, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX)
  DWMH_TC_ATTR(1, true, false, false); DWMH_TC_ATTR(2, true, false, false); DWMH_TC_ATTR(4, true, false, false);
  DWMH_TC_ATTR(1, false, false, false); DWMH_TC_ATTR(2, false, false, false); DWMH_TC_ATTR(4, false, false, false);
  DWMH_TC_ATTR(1, false, true, false); DWMH_TC_ATTR(2, false, true, false); DWMH_TC_ATTR(4, false, true, false);
  DWMH_TC_ATTR(1, true, false, true); DWMH_TC_ATTR(2, true, false, true); DWMH_TC_ATTR(4, true, false, true);
  DWMH_TC_ATTR(1, false, false, true); DWMH_TC_ATTR(2, false, false, true); DWMH_TC_ATTR(4, false, false, true);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3_tc_kernel<T, 2, true, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3_tc_kernel<T, 2, true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3_tc_kernel<T, 2, true, false, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3_tc_kernel<T, 2, true, false, true, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX);
#undef DWMH_TC_ATTR
  return e == cudaSuccess ? 0 : 1;
}

inline int tc_init_attributes(bool bf16) { return bf16 ? tc_set_attr_all<__nv_bfloat16>() : tc_set_attr_all<__half>(); }

struct TcXform { const double* sums; const float* gamma; const float* beta; double inv_count; const void* src; };
// mstride: floats between two modalities of the source (read only by the multi-modality kernel)
struct TcFirstSrc { const float* src; const SampleMeta* metas; int patch_mode, SY, SZ; int64_t mstride; };

// planes per z-block: split D until the grid fills the machine about twice
inline int tc_plan_zb(const TcKParams& kp, int nb, int num_sms) {
  const int tiles = kp.tilesH * kp.tilesW;
  if (!kp.first && !kp.tconv && kp.D >= 16) {
    // 3-D convs on >= 16 planes: minimise waves x input planes per CTA (block + depth halo).  16^3 layers then run 128 CTAs of 18
    // planes in one wave instead of 256 CTAs of 10 planes in two, dec3-a 1024 CTAs in 7 waves instead of 512 in 4 (3.46 rounded up):
    // -6 % on dec3-a, -5..9 % on the 16^3 and the strided layers (profiles/ab_loader_r02b.txt).  The first conv, the transposed
    // convs and the layers on <= 8 planes were faster with the fill rule below.
    const int halo = kp.Jhi - kp.Jlo;
    int best = kp.D; long long best_cost = -1;
    for (int nzb = 1; nzb <= kp.D / 2; ++nzb) {
      const int ZB = (kp.D + nzb - 1) / nzb;
      if ((kp.D + ZB - 1) / ZB != nzb) continue;
      const long long items = (long long)nb * kp.ncb * tiles * nzb;
      const long long ctas = (items + kp.G - 1) / kp.G, waves = (ctas + num_sms - 1) / num_sms;
      const long long cost = waves * (ZB + halo);
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = ZB; }
    }
    return best;
  }
  // split D until the grid fills the machine about twice
  int ZB = kp.D;
  while ((long long)nb * kp.ncb * tiles * ((kp.D + ZB - 1) / ZB) < 2LL * num_sms && ZB > 2) ZB = (ZB + 1) / 2;
  return ZB;
}

// StatPartial entries one launch of this layer writes (0 for a transposed conv): [item][CB]
inline size_t tc_partials_needed(const TcKParams& kp, int nb, int num_sms) {
  if (kp.tconv) return 0;
  const int ZB = tc_plan_zb(kp, nb, num_sms);
  return (size_t)nb * kp.ncb * ((kp.D + ZB - 1) / ZB) * kp.tilesH * kp.tilesW * kp.CB;
}

// sums: the layer's [n][Cout][2] fp64 statistics ({mean, variance} on return); partials: scratch of tc_partials_needed() entries
template <typename T>
int tc_launch(TcLayer& t, int nb, double* sums, StatPartial* partials, int num_sms, cudaStream_t st, std::string* err, const TcXform* xf = nullptr, const TcFirstSrc* fs = nullptr) {
  TcKParams kp = t.kp;
  kp.partials = partials;
  if (!kp.tconv && (!sums || !partials)) { if (err) *err = "conv launch without a statistics buffer"; return 1; }
  if (kp.first) {
    if (!fs) { if (err) *err = "first-conv launch without a source"; return 1; }
    kp.fc_src = fs->src; kp.fc_metas = fs->metas; kp.fc_patch_mode = fs->patch_mode; kp.fc_SY = fs->SY; kp.fc_SZ = fs->SZ;
    kp.fc_mstride = fs->mstride;
  }
  if (xf && t.xform_ok) { kp.xform = 1; kp.xf_sums = xf->sums; kp.xf_gamma = xf->gamma; kp.xf_beta = xf->beta; kp.xf_inv_count = xf->inv_count; kp.xf_src = xf->src; }
  const int tiles = kp.tilesH * kp.tilesW;
  const int ZB = tc_plan_zb(kp, nb, num_sms);
  kp.ZB = ZB; kp.nzb = (kp.D + ZB - 1) / ZB;
  const long long items = (long long)nb * kp.ncb * kp.nzb * tiles;
  // both groups of a CTA must share the cout block whose weights are resident: pairs (2k, 2k+1) stay inside
  // one (n, cb) when the tiles x z-blocks count is even
  if (!kp.first && kp.G == 2 && (kp.resident ? ((long long)kp.nzb * tiles) % 2 != 0 : tiles % 2 != 0)) kp.G = 1;    // (streamed weights: same z-block too)
  kp.total_items = (int)items;
  const unsigned grid = (unsigned)((items + kp.G - 1) / kp.G);
  const unsigned threads = TC_THREADS * kp.G;
  const int ks = kp.KC / 16;
  const bool small = kp.CB <= 32 && !kp.tconv;
#define DWMH_TC_LAUNCH(K, S, C, D) conv3_tc_kernel<T, K, S, C, D, false><<<grid, threads, t.smem_bytes, st>>>(t.tm0, t.tm1, kp)
#define DWMH_TC_LAUNCH_K(S, C, D) do { if (ks == 1) DWMH_TC_LAUNCH(1, S, C, D); else if (ks == 2) DWMH_TC_LAUNCH(2, S, C, D); else DWMH_TC_LAUNCH(4, S, C, D); } while (0)
  if (kp.first && kp.fc_M > 1) conv3_tc_kernel<T, 2, true, false, true, false, true, true><<<grid, 512, t.smem_bytes, st>>>(t.tm0, t.tm1, kp);
  else if (kp.first) conv3_tc_kernel<T, 2, true, false, true, false, true><<<grid, 512, t.smem_bytes, st>>>(t.tm0, t.tm1, kp);
  else if (kp.xform) {
    const unsigned xthreads = (TC_THREADS + 32) * kp.G;
    if (kp.G == 2) conv3_tc_kernel<T, 2, true, false, true, true><<<grid, xthreads, t.smem_bytes, st>>>(t.tm0, t.tm1, kp);
    else conv3_tc_kernel<T, 2, true, false, false, true><<<grid, xthreads, t.smem_bytes, st>>>(t.tm0, t.tm1, kp);
  } else if (kp.tconv) DWMH_TC_LAUNCH_K(false, true, false);
  else if (kp.G == 2) { if (small) DWMH_TC_LAUNCH_K(true, false, true); else DWMH_TC_LAUNCH_K(false, false, true); }
  else { if (small) DWMH_TC_LAUNCH_K(true, false, false); else DWMH_TC_LAUNCH_K(false, false, false); }
#undef DWMH_TC_LAUNCH_K
#undef DWMH_TC_LAUNCH
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { if (err) *err = std::string("conv3_tc_kernel launch failed: ") + cudaGetErrorString(e); return 1; }
  if (!kp.tconv) {
    const int jn = std::max(1, 256 / kp.CB);
    stats_reduce_kernel<<<nb * kp.ncb, kp.CB * jn, 0, st>>>(partials, sums, kp.ncb, kp.CB, kp.Cout, kp.nzb * tiles, jn);
    e = cudaGetLastError();
    if (e != cudaSuccess) { if (err) *err = std::string("stats_reduce_kernel launch failed: ") + cudaGetErrorString(e); return 1; }
  }
  return 0;
}

}  // namespace dwmh
