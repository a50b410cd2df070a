// SURVEY.md section 8f-2: `remove_sparks` of deepwmh/analysis/image_ops.py:325-344 on the device.
// 3-D connected components with 6-connectivity (scipy.ndimage.label's default structuring element) by lock-free
// union-find on voxel indices, then a component-size filter.  Integer work: the result is bit-identical to the
// reference's loop (components smaller than min_volume voxels are discarded, the rest become 1).
// The same labelling serves nnU-Net's postprocessing.json (keep the largest component of a class set, DESIGN §11).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dwmh {

__device__ __forceinline__ int ccl_find(const int* __restrict__ L, int x) {
  int p = L[x];
  while (p != x) { x = p; p = L[x]; }
  return x;
}

// attach the larger root to the smaller one; atomicMin keeps concurrent unions consistent
__device__ __forceinline__ void ccl_union(int* L, int a, int b) {
  while (true) {
    a = ccl_find(L, a);
    b = ccl_find(L, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }
    const int old = atomicMin(&L[a], b);
    if (old == a) return;
    a = old;
  }
}

// Run pre-linking: consecutive lanes hold consecutive voxels of a z-row, so one ballot tells every foreground voxel where
// its run starts inside the warp's 32-voxel segment; labels start out as that run start (trees of depth 1) and the merge
// pass only has to stitch runs across segment boundaries and across rows / planes.  `fg` must be evaluated by all 32 lanes.
__device__ __forceinline__ int ccl_run_start(bool fg, bool row_start, int64_t v) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned fgm = __ballot_sync(0xffffffffu, fg);
  const unsigned brk = __ballot_sync(0xffffffffu, fg && (lane == 0 || row_start || !((fgm >> (lane - 1)) & 1u)));
  if (!fg) return -1;
  const unsigned upto = brk & (0xffffffffu >> (31u - lane));        // breaks at lanes <= this one
  return (int)(v - (int64_t)(lane - (31u - __clz(upto))));
}

// mask: voxel > 0 (uint8 label map) ; labels[v] = start of v's z-run (within its 32-voxel segment), -1 for background
static __global__ void __launch_bounds__(256) ccl_init_kernel(const uint8_t* __restrict__ seg, int* __restrict__ L, int* __restrict__ size,
                                                              int64_t V, int Z) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); v0 < V; v0 += stride) {   // warp-uniform trip count
    const int64_t v = v0 + (threadIdx.x & 31);
    const bool in = v < V;
    const int l = ccl_run_start(in && seg[v] != 0, in && v % Z == 0, v);
    if (in) { L[v] = l; size[v] = 0; }
  }
}

static __global__ void __launch_bounds__(256) ccl_merge_kernel(int* __restrict__ L, int X, int Y, int Z) {
  const int64_t V = (int64_t)X * Y * Z;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) {
    if (L[v] < 0) continue;
    const int z = (int)(v % Z), y = (int)((v / Z) % Y), x = (int)(v / ((int64_t)Z * Y));
    if (((v + 1) & 31) == 0 && z + 1 < Z && L[v + 1] >= 0) ccl_union(L, (int)v, (int)v + 1);   // inside a segment the runs are linked already
    if (y + 1 < Y && L[v + Z] >= 0) ccl_union(L, (int)v, (int)(v + Z));
    if (x + 1 < X && L[v + (int64_t)Z * Y] >= 0) ccl_union(L, (int)v, (int)(v + (int64_t)Z * Y));
  }
}

static __global__ void __launch_bounds__(256) ccl_count_kernel(int* __restrict__ L, int* __restrict__ size, int64_t V) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) {
    if (L[v] < 0) continue;
    const int r = ccl_find(L, (int)v);
    L[v] = r;                                   // safe: roots never change after the merge pass
    atomicAdd(&size[r], 1);
  }
}

static __global__ void __launch_bounds__(256) ccl_filter_kernel(const int* __restrict__ L, const int* __restrict__ size, uint8_t* __restrict__ out,
                                                         int min_volume, int64_t V) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) {
    const int r = L[v];
    out[v] = (r >= 0 && size[r] >= min_volume) ? 1 : 0;
  }
}

// ---- nnU-Net v1 postprocessing (remove_all_but_the_largest_connected_component), one entry of postprocessing.json ----
// The mask is class-set membership: bit seg[v] of class_mask (labels >= 32 are never in the set).  Same labels as
// ccl_init_kernel otherwise, so ccl_merge_kernel / ccl_count_kernel run unchanged.  Also clears the maximum for this call.
static __global__ void __launch_bounds__(256) ccl_init_classes_kernel(const uint8_t* __restrict__ seg, int* __restrict__ L, int* __restrict__ size,
                                                                      int* __restrict__ max_size, uint32_t class_mask, int64_t V, int Z) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *max_size = 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); v0 < V; v0 += stride) {   // warp-uniform trip count
    const int64_t v = v0 + (threadIdx.x & 31);
    const bool in = v < V;
    const unsigned s = in ? seg[v] : 32u;
    const int l = ccl_run_start(s < 32u && ((class_mask >> s) & 1u), in && v % Z == 0, v);
    if (in) { L[v] = l; size[v] = 0; }
  }
}

// largest component: size[] is non-zero at roots only; integer max, so the result does not depend on the order
static __global__ void __launch_bounds__(256) ccl_max_size_kernel(const int* __restrict__ size, int* __restrict__ max_size, int64_t V) {
  int m = 0;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) m = max(m, size[v]);
  for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(max_size, m);
}

// Zero the voxels of the mask whose component is not of the largest size and, when min_valid_mm3 >= 0, is smaller than
// min_valid_mm3 (count * volume_per_voxel in fp64, as upstream compares its sizes).  Voxels outside the mask are not written.
static __global__ void __launch_bounds__(256) ccl_keep_largest_kernel(const int* __restrict__ L, const int* __restrict__ size,
                                                                      const int* __restrict__ max_size, uint8_t* __restrict__ seg,
                                                                      double volume_per_voxel, double min_valid_mm3, int64_t V) {
  const int keep = *max_size;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) {
    const int r = L[v];
    if (r < 0) continue;
    const int n = size[r];
    if (n == keep) continue;
    if (min_valid_mm3 >= 0.0 && (double)n * volume_per_voxel >= min_valid_mm3) continue;
    seg[v] = 0;
  }
}

}  // namespace dwmh
