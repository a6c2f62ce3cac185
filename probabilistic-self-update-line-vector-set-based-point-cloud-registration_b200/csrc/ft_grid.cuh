// ft_grid.cuh -- FPFH's grid over a batch of raw clouds (k8_features.cu: normals and FPFH; k8_colors.cu: the colour
// gradients of colored ICP): FP32 cells of size h hashed into each cloud's bucket table, the build kernels that sort
// every bucket's members by index, the 27-cell neighbour walks and the hybrid (radius + max_nn) selection.
#pragma once

#include <cuda_runtime.h>

#include <vector>

#include "common.cuh"
#include "ft_batch.cuh"
#include "grid.cuh"

namespace psulvsb {

namespace {

struct Grid {
  double inv_h;
  unsigned int mask;  // nb - 1
  const float4* spts;     // [n] sorted by bucket, ascending index inside a bucket; .w = index bits
  const int* start;       // [nb + 1]
};

__device__ __forceinline__ long long cell_of(float x, double inv_h) { return (long long)floor((double)x * inv_h); }

// FP32 squared distance, left to right and unfused (the restatement evaluates the same expression in numpy float32)
__device__ __forceinline__ float sqdist(float4 a, float4 b) {
  const float dx = b.x - a.x, dy = b.y - a.y, dz = b.z - a.z;
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// Calls f(q, j) for every point q (float4, .w = index bits) with |q - p|^2 <= r2 in FP32 (p itself included).
template <typename F>
__device__ __forceinline__ void for_neighbours(const Grid& g, float4 p, float r2, F f) {
  const long long cx = cell_of(p.x, g.inv_h), cy = cell_of(p.y, g.inv_h), cz = cell_of(p.z, g.inv_h);
  unsigned int seen[27];
  int ns = 0;
  for (int dz = -1; dz <= 1; ++dz)
    for (int dy = -1; dy <= 1; ++dy)
      for (int dx = -1; dx <= 1; ++dx) {
        const unsigned int b = bucket_of(cx + dx, cy + dy, cz + dz, g.mask);
        bool dup = false;
        for (int s = 0; s < ns; ++s) dup |= seen[s] == b;
        if (dup) continue;
        seen[ns++] = b;
        const int e = g.start[b + 1];
        for (int t = g.start[b]; t < e; ++t) {
          const float4 q = g.spts[t];
          if (sqdist(p, q) <= r2) f(q, __float_as_int(q.w));
        }
      }
}

// for_neighbours' walk without its local array, so that a kernel keeps no stack frame: the same 27 cells in the same
// order, each bucket once (visit bit k = the first cell of its bucket)
template <typename F>
__device__ __forceinline__ void for_neighbours_masked(const Grid& g, float4 p, float r2, F f) {
  const long long cx = cell_of(p.x, g.inv_h), cy = cell_of(p.y, g.inv_h), cz = cell_of(p.z, g.inv_h);
  unsigned int visit = 0;
  {
    unsigned int b[27];
#pragma unroll
    for (int k = 0; k < 27; ++k) {
      b[k] = bucket_of(cx + k % 3 - 1, cy + (k / 3) % 3 - 1, cz + k / 9 - 1, g.mask);
      bool dup = false;
#pragma unroll
      for (int s = 0; s < k; ++s) dup |= b[s] == b[k];
      if (!dup) visit |= 1u << k;
    }
  }
#pragma unroll 1
  for (int k = 0; k < 27; ++k) {
    if (!((visit >> k) & 1u)) continue;
    const unsigned int b = bucket_of(cx + k % 3 - 1, cy + (k / 3) % 3 - 1, cz + k / 9 - 1, g.mask);
    const int e = g.start[b + 1];
    for (int t = g.start[b]; t < e; ++t) {
      const float4 q = g.spts[t];
      if (sqdist(p, q) <= r2) f(q, __float_as_int(q.w));
    }
  }
}

// ---- grid build: count, scan (one CTA per cloud), scatter (grid.cuh), order (each bucket's members ascending by index)
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS)
    k8_grid_count(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one, const int* __restrict__ tile_first, int B, double inv_h,
                  int* __restrict__ pbucket, int* __restrict__ count) {
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int i = first + threadIdx.x;
  if (i >= cl.n) return;
  const double* pts = cl.pts;
  const float x = (float)pts[3 * (size_t)i], y = (float)pts[3 * (size_t)i + 1], z = (float)pts[3 * (size_t)i + 2];
  const int b = cl.b0 + (int)bucket_of(cell_of(x, inv_h), cell_of(y, inv_h), cell_of(z, inv_h), cl.mask);
  pbucket[cl.p0 + i] = b;
  atomicAdd(count + b, 1);
}

// the scatter's order inside a bucket depends on timing: rank each member by index instead
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS)
    k8_grid_order(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one, const int* __restrict__ tile_first, int B,
                  const int* __restrict__ pbucket, const int* __restrict__ start, const int* __restrict__ tmp,
                  float4* __restrict__ spts) {
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int l = first + threadIdx.x;
  if (l >= cl.n) return;
  const int i = tmp[cl.p0 + l];
  const int b = pbucket[i] + ci, s0 = start[b], s1 = start[b + 1];
  int rank = 0;
  for (int q = s0; q < s1; ++q) rank += tmp[q] < i;
  const int j = i - cl.p0;
  const double* pts = cl.pts;
  spts[s0 + rank] = make_float4((float)pts[3 * (size_t)j], (float)pts[3 * (size_t)j + 1], (float)pts[3 * (size_t)j + 2],
                                __int_as_float(j));
}

// hybrid normals: candidate j of point p ranks by (FP32 |p_j - p|^2 bits, j); d^2 >= 0, so the bits keep its order
constexpr int FT_MAX_NN = 32;

__device__ __forceinline__ unsigned long long nn_key(float4 p, float4 q, int j) {
  return ((unsigned long long)__float_as_uint(sqdist(p, q)) << 32) | (unsigned int)j;
}

// the hybrid neighbourhood of `me`: a walk over the points within r2 (for_neighbours, or for_neighbours_masked with
// kMasked) keeps the max_nn smallest keys in the kernel's shared `kept` (column tid; [slot][thread]: a warp's slot s is
// 32 consecutive words).  kstar = the max_nn-th smallest key, or ~0 (every key) when the neighbourhood is no larger;
// nk = the neighbourhood's size.  A later walk that skips keys above kstar visits the kept points in the radius walk's
// order.  (The kernel passes threadIdx.x: read here, it changes k8_radius_normals' instruction selection.)
struct Hybrid {
  unsigned long long kstar;
  int nk;
};
template <bool kMasked>
__device__ __forceinline__ Hybrid hybrid_threshold(const Grid& g, float4 me, float r2, int max_nn,
                                                   unsigned long long (&kept)[FT_MAX_NN][FT_THREADS], int tid) {
  int nk = 0, top = 0;  // candidates seen; the slot of the largest kept key
  unsigned long long kmax = 0;
  auto keep = [&](float4 q, int j) {
    const unsigned long long k = nn_key(me, q, j);
    if (nk < max_nn) {
      kept[nk][tid] = k;
      if (k > kmax) {
        kmax = k;
        top = nk;
      }
    } else if (k < kmax) {  // replace the largest, then find the new largest
      kept[top][tid] = k;
      kmax = 0;
      for (int s = 0; s < max_nn; ++s) {
        const unsigned long long v = kept[s][tid];
        if (v > kmax) {
          kmax = v;
          top = s;
        }
      }
    }
    ++nk;
  };
  if constexpr (kMasked)
    for_neighbours_masked(g, me, r2, keep);
  else
    for_neighbours(g, me, r2, keep);
  return Hybrid{nk > max_nn ? kmax : ~0ull, nk};
}

// the batch's table: FtCloud[B], then tile_first[B + 1]
std::vector<char> cloud_table(const psulvsb_fpfh_cloud_t* clouds, int B, size_t table_bytes) {
  std::vector<char> table(table_bytes);
  FtCloud* hc = reinterpret_cast<FtCloud*>(table.data());
  int* tile_first = reinterpret_cast<int*>(table.data() + sizeof(FtCloud) * (size_t)B);
  tile_first[0] = 0;
  long long p0 = 0, b0 = 0;
  for (int c = 0; c < B; ++c) {
    const psulvsb_fpfh_cloud_t& q = clouds[c];
    FtCloud& h = hc[c];
    const unsigned int nb = q.n > 0 ? bucket_count(q.n) : 0u;
    h.pts = q.pts;
    for (int r = 0; r < 3; ++r) h.vp[r] = q.viewpoint[r];
    h.n = q.n;
    h.p0 = (int)p0;
    h.b0 = (int)b0;
    h.mask = nb - 1;
    p0 += q.n;
    b0 += nb;
    tile_first[c + 1] = tile_first[c] + blocks(q.n, FT_THREADS);
  }
  return table;
}

}  // namespace

}  // namespace psulvsb
