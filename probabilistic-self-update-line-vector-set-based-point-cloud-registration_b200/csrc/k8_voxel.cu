// k8_voxel.cu -- the voxel-grid filter (Open3D's PointCloud::VoxelDownSample), single and batched.  The pipeline, on
// the FPFH stage's batch table and hashed grid, is ft_voxel.cuh's; this file holds its mean pass and the C ABI.
// DESIGN.md section 10, "Voxel downsampling", is the specification; tests/voxel_restatement.py restates it in numpy.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "ft_batch.cuh"
#include "ft_voxel.cuh"
#include "grid.cuh"

namespace psulvsb {

namespace {

// ---- each representative takes the column tile offset + its rank in the tile and writes the mean of the members of
// its bucket with its cell, walking the bucket from its own sorted position (no earlier member has the cell)
// (ptxas otherwise caps the batch instantiation at 32 registers and spills)
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS, 8)
    k8_voxel_mean(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one,
                  const int* __restrict__ tile_first, int B, const int* __restrict__ pbucket,
                  const int* __restrict__ start, const int* __restrict__ spos, const int* __restrict__ sidx,
                  const Cell* __restrict__ scell, const unsigned char* __restrict__ rep,
                  const int* __restrict__ tile_start, double* __restrict__ out) {
  __shared__ int warp_n[FT_THREADS / 32];
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const double* pts = cl.pts;
  const int p0 = cl.p0;
  const int i = first + threadIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const size_t o = (size_t)p0 + i;
  const bool r = i < cl.n && rep[o];
  const unsigned int bal = __ballot_sync(0xffffffffu, r);
  if (lane == 0) warp_n[wid] = __popc(bal);
  __syncthreads();
  if (!r) return;
  int slot = tile_start[blockIdx.x + ci] + __popc(bal & ((1u << lane) - 1u));
  for (int w = 0; w < wid; ++w) slot += warp_n[w];
  const int s = spos[o], s1 = start[pbucket[o] + ci + 1];
  const Cell c = scell[s];
  double sx = 0.0, sy = 0.0, sz = 0.0;
  int cnt = 0;
  for (int t = s; t < s1; ++t) {
    if (!same_cell(scell[t], c)) continue;
    const size_t j = (size_t)sidx[t];
    sx += pts[3 * j];
    sy += pts[3 * j + 1];
    sz += pts[3 * j + 2];
    ++cnt;
  }
  const size_t d = (size_t)p0 + slot;
  out[3 * d] = sx / (double)cnt;
  out[3 * d + 1] = sy / (double)cnt;
  out[3 * d + 2] = sz / (double)cnt;
}

// the batch on the device (clouds checked, B >= 1): one upload of the cloud table (batches only), one memset, eight
// launches over all clouds; every count is written on the device
int run_voxel(cudaStream_t st, const psulvsb_fpfh_cloud_t* clouds, int B, double v, void* work, double* out,
              int* counts) {
  return run_voxel_passes(st, clouds, B, v, work, counts, [&](auto batch, const VoxelWork& w, const FtCloud& one,
                                                              int tiles) -> int {
    k8_voxel_mean<decltype(batch)::value><<<tiles, FT_THREADS, 0, st>>>(
        w.cloud, one, w.tile_first, B, w.pbucket, w.start, w.spos, w.sidx, w.scell, w.rep, w.tile_start, out);
    return PSULVSB_OK;
  });
}

// the batch on host buffers (clouds checked, B >= 1): the clouds go up in one copy, the counts and the voxels come back
int run_voxel_host(const psulvsb_fpfh_cloud_t* clouds, int B, double v, double* out, int* counts, const char* who) {
  const FpfhSizes z = fpfh_sizes(clouds, B);
  if (z.n == 0) {
    std::memset(counts, 0, sizeof(int) * (size_t)B);
    return PSULVSB_OK;
  }
  const size_t N = (size_t)z.n, o_c = up256(24 * N), o_in = o_c + up256(4 * (size_t)B), o_w = o_in + up256(24 * N);
  std::vector<char> in(B > 1 ? 24 * N : 0);
  std::vector<psulvsb_fpfh_cloud_t> dev(clouds, clouds + B);
  DevBuf buf;
  if (int rc = buf.alloc(o_w + voxel_layout(z, nullptr, nullptr), who)) return rc;
  char* b = static_cast<char*>(buf.p);
  // a single cloud goes up straight from the caller's buffer: packing it first would only add a host copy
  size_t off = 0;
  for (int c = 0; c < B; ++c) {
    if (dev[c].n <= 0) continue;
    const size_t bytes = 24 * (size_t)dev[c].n;
    if (B > 1) std::memcpy(in.data() + off, dev[c].pts, bytes);
    dev[c].pts = reinterpret_cast<const double*>(b + o_in + off);
    off += bytes;
  }
  PSU_CUDA(cudaMemcpyAsync(b + o_in, B > 1 ? in.data() : (const void*)clouds[0].pts, 24 * N, cudaMemcpyHostToDevice,
                           nullptr));
  if (int rc = run_voxel(nullptr, dev.data(), B, v, b + o_w, (double*)b, (int*)(b + o_c))) return rc;
  PSU_CUDA(cudaMemcpyAsync(counts, b + o_c, 4 * (size_t)B, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaMemcpyAsync(out, b, 24 * N, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaStreamSynchronize(nullptr));
  return PSULVSB_OK;
}

}  // namespace

}  // namespace psulvsb

using psulvsb::fail;

extern "C" {

// ---- voxel downsampling (DESIGN.md section 10, "Voxel downsampling")
unsigned long long psulvsb_voxel_down_sample_workspace_bytes(int n) {
  if (n < 0) return 0ull;
  const psulvsb_fpfh_cloud_t c{nullptr, n, {0.0, 0.0, 0.0}};
  return (unsigned long long)psulvsb::voxel_layout(psulvsb::fpfh_sizes(&c, 1), nullptr, nullptr);
}

unsigned long long psulvsb_voxel_down_sample_batch_workspace_bytes(const psulvsb_fpfh_cloud_t* clouds, int B) {
  if (B <= 0 || !clouds) return 0ull;
  for (int c = 0; c < B; ++c)
    if (clouds[c].n < 0) return 0ull;
  return (unsigned long long)psulvsb::voxel_layout(psulvsb::fpfh_sizes(clouds, B), nullptr, nullptr);
}

int psulvsb_voxel_down_sample(void* stream, const double* d_pts, int n, double voxel_size, void* d_work,
                              double* d_out, int* d_count) {
  if (n < 0 || !psulvsb::voxel_ok(voxel_size) || !d_count || (n > 0 && (!d_pts || !d_work || !d_out)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_voxel_down_sample: bad argument (voxel_size must be finite and > 0)");
  const psulvsb_fpfh_cloud_t c{d_pts, n, {0.0, 0.0, 0.0}};
  if (int rc = psulvsb::clouds_check(&c, 1, "psulvsb_voxel_down_sample")) return rc;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_voxel((cudaStream_t)stream, &c, 1, voxel_size, d_work, d_out, d_count);
}

int psulvsb_voxel_down_sample_host(const double* pts, int n, double voxel_size, double* out, int* n_out) {
  if (n < 0 || !psulvsb::voxel_ok(voxel_size) || !n_out || (n > 0 && (!pts || !out)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_voxel_down_sample_host: bad argument (voxel_size must be finite and > 0)");
  *n_out = 0;
  const psulvsb_fpfh_cloud_t c{pts, n, {0.0, 0.0, 0.0}};
  if (int rc = psulvsb::clouds_check(&c, 1, "psulvsb_voxel_down_sample_host")) return rc;
  if (n == 0) return PSULVSB_OK;  // the zero count is written on the host: no device needed
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_voxel_host(&c, 1, voxel_size, out, n_out, "psulvsb_voxel_down_sample_host");
}

int psulvsb_voxel_down_sample_batch(void* stream, const psulvsb_fpfh_cloud_t* clouds, int B, double voxel_size,
                                    void* d_work, double* d_out, int* d_counts) {
  if (B < 0 || !psulvsb::voxel_ok(voxel_size) || (B > 0 && (!clouds || !d_work || !d_out || !d_counts)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_voxel_down_sample_batch: bad argument (voxel_size must be finite and > 0)");
  if (int rc = psulvsb::clouds_check(clouds, B, "psulvsb_voxel_down_sample_batch")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_voxel((cudaStream_t)stream, clouds, B, voxel_size, d_work, d_out, d_counts);
}

int psulvsb_voxel_down_sample_batch_host(const psulvsb_fpfh_cloud_t* clouds, int B, double voxel_size, double* out,
                                         int* counts) {
  if (B < 0 || !psulvsb::voxel_ok(voxel_size) || (B > 0 && (!clouds || !out || !counts)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_voxel_down_sample_batch_host: bad argument (voxel_size must be finite and > 0)");
  if (int rc = psulvsb::clouds_check(clouds, B, "psulvsb_voxel_down_sample_batch_host")) return rc;
  if (psulvsb::fpfh_sizes(clouds, B).n == 0) {  // zero counts, written on the host: no device needed
    std::memset(counts, 0, sizeof(int) * (size_t)B);
    return PSULVSB_OK;
  }
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_voxel_host(clouds, B, voxel_size, out, counts, "psulvsb_voxel_down_sample_batch_host");
}

}  // extern "C"
