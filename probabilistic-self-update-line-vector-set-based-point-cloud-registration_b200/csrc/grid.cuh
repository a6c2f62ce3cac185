// grid.cuh -- the hashed uniform grid shared by the FPFH stage (k8_features.cu) and ICP (k9_icp.cu): the bucket hash,
// the one-CTA exclusive scan of the bucket counts (both scan one segment per cloud of a batch with it), the scatter of
// point indices into their buckets and the lookup of a batch item by its prefix.  Each user bins
// its own coordinates (FP32 cells for FPFH, FP64 cells relative to the bounding-box corner for ICP) and orders each
// bucket's members by index itself, so a bucket's points sit in ascending index order whatever the scatter's timing.
#pragma once

#include <cuda_runtime.h>

namespace psulvsb {

namespace {

constexpr int SCAN_THREADS = 1024;
constexpr int GRID_THREADS = 128;

// nb = 2^ceil(log2 n) buckets (at least one): the workspace depends on n only
inline unsigned int bucket_count(int n) {
  unsigned int nb = 1;
  while (nb < (unsigned int)n) nb <<= 1;
  return nb;
}

__device__ __forceinline__ unsigned int bucket_of(long long cx, long long cy, long long cz, unsigned int mask) {
  unsigned long long k = (unsigned long long)cx * 0x9E3779B97F4A7C15ull ^ (unsigned long long)cy * 0xC2B2AE3D27D4EB4Full ^
                         (unsigned long long)cz * 0x165667B19E3779F9ull;
  k ^= k >> 31;
  k *= 0xBF58476D1CE4E5B9ull;
  k ^= k >> 29;
  return (unsigned int)k & mask;
}

// base + exclusive scan of count[0, m) into start[0, m] by one CTA of SCAN_THREADS threads, and cursor = start
__device__ __forceinline__ void cta_scan(const int* __restrict__ count, int m, int* __restrict__ start,
                                         int* __restrict__ cursor, int base) {
  __shared__ int warp_tot[SCAN_THREADS / 32];
  __shared__ int carry;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) carry = base;
  __syncthreads();
  for (int i0 = 0; i0 < m; i0 += SCAN_THREADS) {
    const int i = i0 + tid;
    const int v = i < m ? count[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[wid] = x;
    __syncthreads();
    if (wid == 0) {
      int w = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      warp_tot[lane] = w;
    }
    __syncthreads();
    const int excl = carry + (wid ? warp_tot[wid - 1] : 0) + x - v;
    if (i < m) {
      start[i] = excl;
      if (cursor) cursor[i] = excl;
    }
    __syncthreads();
    if (tid == 0) carry += warp_tot[SCAN_THREADS / 32 - 1];
    __syncthreads();
  }
  if (tid == 0) start[m] = carry;
}

// the item of x in a batch: the p with first[p] <= x < first[p + 1] (first[0, B] ascending, first[0] <= x < first[B]; an
// item without entries is never the answer)
__device__ __forceinline__ int pair_of(const int* __restrict__ first, int B, int x) {
  int lo = 0, hi = B;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (first[mid] <= x)
      lo = mid;
    else
      hi = mid;
  }
  return lo;
}

// tmp[start[b] ..] receives the indices of bucket b's members in arrival order; a point with a negative bucket is left
// out of the grid
__global__ void __launch_bounds__(GRID_THREADS)
    k8_grid_scatter(int n, const int* __restrict__ pbucket, int* __restrict__ cursor, int* __restrict__ tmp) {
  const int i = blockIdx.x * GRID_THREADS + threadIdx.x;
  if (i >= n) return;
  const int b = pbucket[i];
  if (b >= 0) tmp[atomicAdd(cursor + b, 1)] = i;
}

}  // namespace

}  // namespace psulvsb
