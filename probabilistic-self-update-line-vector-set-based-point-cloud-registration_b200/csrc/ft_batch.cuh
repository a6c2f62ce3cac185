// ft_batch.cuh -- the batch table of the raw-cloud stages on FPFH's grid (k8_features.cu: FPFH and normals;
// k8_voxel.cu: the voxel filter): one cloud per item, each starting on a 128-point tile with its own bucket table; the
// per-cloud scan of the bucket counts; the host-side sizes, workspace helpers and the check of a batch's clouds.
#pragma once

#include <cuda_runtime.h>

#include <string>

#include "common.cuh"
#include "grid.cuh"

namespace psulvsb {

namespace {

constexpr int FT_THREADS = 128;

// ---- batches (FPFH, normals, voxel filter).  Every cloud starts on a 128-point tile, so a CTA belongs to one cloud;
// it finds it by pair_of over the prefix of the clouds' tiles.  Per-point arrays (spts, nf, pbucket, tmp, counts,
// kcount, the outputs) are the concatenation of the clouds' (cloud c's from p0); each cloud keeps its own table of
// bucket_count(n) buckets, whose start entries count positions from the batch's first point.
struct FtCloud {
  const double* pts;  // 3 x n, column-major
  double vp[3];       // normals flip towards it (the voxel filter has no normals)
  int n;
  int p0;             // first point in the per-point arrays
  int b0;             // first bucket (count, cursor); the start table is start[b0 + c, b0 + c + nb] for cloud c
  unsigned int mask;  // nb - 1
};

// the CTA's cloud ci and the cloud's index of the CTA's first point.  A batch of one (kBatch false) takes its cloud
// from the kernel parameter `one`: its fields stay operands of the parameter bank instead of registers.
template <bool kBatch>
__device__ __forceinline__ const FtCloud& cloud_tile(const FtCloud* __restrict__ clouds, const FtCloud& one,
                                              const int* __restrict__ tile_first, int B, int& ci, int& first) {
  if constexpr (kBatch) {
    ci = pair_of(tile_first, B, blockIdx.x);
    first = (blockIdx.x - tile_first[ci]) * FT_THREADS;
    return clouds[ci];
  } else {
    ci = 0;
    first = blockIdx.x * FT_THREADS;
    return one;
  }
}

template <bool kBatch>
__global__ void __launch_bounds__(SCAN_THREADS)
    k8_cloud_scan(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one, const int* __restrict__ count,
                  int* __restrict__ start, int* __restrict__ cursor) {
  const FtCloud& cl = kBatch ? clouds[blockIdx.x] : one;
  if (cl.n == 0) return;
  cta_scan(count + cl.b0, (int)(cl.mask + 1), start + cl.b0 + blockIdx.x, cursor + cl.b0, cl.p0);
}

inline size_t up256(size_t x) { return (x + 255) & ~size_t(255); }

struct DevBuf {
  void* p = nullptr;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  int alloc(size_t bytes, const char* what) {
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) {
      cudaGetLastError();
      p = nullptr;
      return fail(PSULVSB_ERR_CUDA, std::string(what) + ": cudaMalloc failed");
    }
    return PSULVSB_OK;
  }
};

inline int blocks(long long n, int t) { return (int)((n + t - 1) / t); }

// ---- FPFH batch on the host side
struct FpfhSizes {
  long long n = 0, nb = 0, tiles = 0;
  int B = 0;
};

FpfhSizes fpfh_sizes(const psulvsb_fpfh_cloud_t* clouds, int B) {
  FpfhSizes z;
  z.B = B;
  for (int c = 0; c < B; ++c) {
    const int n = clouds[c].n;
    if (n <= 0) continue;
    z.n += n;
    z.nb += bucket_count(n);
    z.tiles += (n + FT_THREADS - 1) / FT_THREADS;
  }
  return z;
}

// PSULVSB_ERR_INVALID for a bad cloud, PSULVSB_ERR_UNSUPPORTED for concatenations past the int range, else OK
int clouds_check(const psulvsb_fpfh_cloud_t* clouds, int B, const char* who) {
  for (int c = 0; c < B; ++c)
    if (clouds[c].n < 0 || (clouds[c].n > 0 && !clouds[c].pts))
      return fail(PSULVSB_ERR_INVALID, std::string(who) + ": bad cloud " + std::to_string(c));
  const FpfhSizes z = fpfh_sizes(clouds, B);
  if (z.n >= (1ll << 31) || z.nb + B >= (1ll << 31))
    return fail(PSULVSB_ERR_UNSUPPORTED, std::string(who) + ": the batch's clouds exceed 2^31 - 1 points in all");
  return PSULVSB_OK;
}

}  // namespace

}  // namespace psulvsb
