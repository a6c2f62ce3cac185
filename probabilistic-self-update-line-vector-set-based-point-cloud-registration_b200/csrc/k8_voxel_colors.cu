// k8_voxel_colors.cu -- the voxel-grid filter that carries colours (Open3D's PointCloud::VoxelDownSample on a cloud
// with colours), single and batched: ft_voxel.cuh's pipeline, whose mean pass also averages each voxel's colours.
// DESIGN.md section 10, "Voxel downsampling with colours", is the specification; tests/voxel_colors_restatement.py
// restates it in numpy.  The file is apart from k8_voxel.cu, whose kernel set a register test pins.
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

// ---- the mean pass with colours: k8_voxel_mean (k8_voxel.cu), whose member walk also sums the members' colours,
// channel by channel in the same order, with the same division.  Cloud ci's colours are colors[ci] (batches) or
// one_colors (a batch of one).
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS, 8)
    k8_voxel_mean_colors(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one,
                         const double* const* __restrict__ colors, const double* __restrict__ one_colors,
                         const int* __restrict__ tile_first, int B, const int* __restrict__ pbucket,
                         const int* __restrict__ start, const int* __restrict__ spos, const int* __restrict__ sidx,
                         const Cell* __restrict__ scell, const unsigned char* __restrict__ rep,
                         const int* __restrict__ tile_start, double* __restrict__ out,
                         double* __restrict__ out_colors) {
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
  const double* col = kBatch ? colors[ci] : one_colors;
  double sx = 0.0, sy = 0.0, sz = 0.0, sr = 0.0, sg = 0.0, sb = 0.0;
  int cnt = 0;
  for (int t = s; t < s1; ++t) {
    if (!same_cell(scell[t], c)) continue;
    const size_t j = (size_t)sidx[t];
    sx += pts[3 * j];
    sy += pts[3 * j + 1];
    sz += pts[3 * j + 2];
    sr += col[3 * j];
    sg += col[3 * j + 1];
    sb += col[3 * j + 2];
    ++cnt;
  }
  const size_t d = (size_t)p0 + slot;
  out[3 * d] = sx / (double)cnt;
  out[3 * d + 1] = sy / (double)cnt;
  out[3 * d + 2] = sz / (double)cnt;
  out_colors[3 * d] = sr / (double)cnt;
  out_colors[3 * d + 1] = sg / (double)cnt;
  out_colors[3 * d + 2] = sb / (double)cnt;
}

std::vector<psulvsb_fpfh_cloud_t> point_clouds(const psulvsb_color_cloud_t* clouds, int B) {
  std::vector<psulvsb_fpfh_cloud_t> f((size_t)(B > 0 ? B : 0));
  for (int c = 0; c < B; ++c) f[c] = psulvsb_fpfh_cloud_t{clouds[c].points, clouds[c].n, {0.0, 0.0, 0.0}};
  return f;
}

// the plain filter's workspace, followed by the colour side table [B]
size_t colors_workspace(const FpfhSizes& z) { return voxel_layout(z, nullptr, nullptr) + up256(8 * (size_t)z.B); }

// PSULVSB_ERR_INVALID for a bad cloud (a NULL colour array of a non-empty cloud included), PSULVSB_ERR_UNSUPPORTED
// for concatenations past the int range, else OK
int colors_check(const psulvsb_color_cloud_t* clouds, int B, const char* who) {
  for (int c = 0; c < B; ++c)
    if (clouds[c].n > 0 && !clouds[c].colors)
      return fail(PSULVSB_ERR_INVALID, std::string(who) + ": bad cloud " + std::to_string(c) + " (no colours)");
  const std::vector<psulvsb_fpfh_cloud_t> f = point_clouds(clouds, B);
  return clouds_check(f.data(), B, who);
}

// the batch on the device (clouds checked, B >= 1): the plain filter's passes; a batch uploads its colour table after
// the cloud table, a batch of one passes its colours as a kernel argument
int run_voxel_colors(cudaStream_t st, const psulvsb_color_cloud_t* clouds, int B, double v, void* work, double* out,
                     double* out_colors, int* counts) {
  const std::vector<psulvsb_fpfh_cloud_t> f = point_clouds(clouds, B);
  const FpfhSizes z = fpfh_sizes(f.data(), B);
  const double** side = reinterpret_cast<const double**>(static_cast<char*>(work) + voxel_layout(z, nullptr, nullptr));
  std::vector<const double*> hs((size_t)B);
  for (int c = 0; c < B; ++c) hs[c] = clouds[c].colors;
  return run_voxel_passes(st, f.data(), B, v, work, counts, [&](auto batch, const VoxelWork& w, const FtCloud& one,
                                                                int tiles) -> int {
    if (B > 1) PSU_CUDA(cudaMemcpyAsync(side, hs.data(), 8 * (size_t)B, cudaMemcpyHostToDevice, st));
    k8_voxel_mean_colors<decltype(batch)::value><<<tiles, FT_THREADS, 0, st>>>(
        w.cloud, one, side, hs[0], w.tile_first, B, w.pbucket, w.start, w.spos, w.sidx, w.scell, w.rep, w.tile_start,
        out, out_colors);
    return PSULVSB_OK;
  });
}

// the batch on host buffers (clouds checked, B >= 1): points and colours go up in one copy; the counts, the voxels and
// their colours come back
int run_voxel_colors_host(const psulvsb_color_cloud_t* clouds, int B, double v, double* out, double* out_colors,
                          int* counts, const char* who) {
  const std::vector<psulvsb_fpfh_cloud_t> f = point_clouds(clouds, B);
  const FpfhSizes z = fpfh_sizes(f.data(), B);
  if (z.n == 0) {
    std::memset(counts, 0, sizeof(int) * (size_t)B);
    return PSULVSB_OK;
  }
  const size_t N = (size_t)z.n, o_oc = up256(24 * N), o_c = o_oc + up256(24 * N), o_in = o_c + up256(4 * (size_t)B),
               o_w = o_in + up256(48 * N);
  std::vector<char> in(48 * N);
  std::vector<psulvsb_color_cloud_t> dev(clouds, clouds + B);
  DevBuf buf;
  if (int rc = buf.alloc(o_w + colors_workspace(z), who)) return rc;
  char* b = static_cast<char*>(buf.p);
  size_t off = 0;
  for (int c = 0; c < B; ++c) {
    if (dev[c].n <= 0) continue;
    const size_t bytes = 24 * (size_t)dev[c].n;
    std::memcpy(in.data() + off, dev[c].points, bytes);
    std::memcpy(in.data() + 24 * N + off, dev[c].colors, bytes);
    dev[c].points = reinterpret_cast<const double*>(b + o_in + off);
    dev[c].colors = reinterpret_cast<const double*>(b + o_in + 24 * N + off);
    off += bytes;
  }
  PSU_CUDA(cudaMemcpyAsync(b + o_in, in.data(), in.size(), cudaMemcpyHostToDevice, nullptr));
  if (int rc = run_voxel_colors(nullptr, dev.data(), B, v, b + o_w, (double*)b, (double*)(b + o_oc), (int*)(b + o_c)))
    return rc;
  PSU_CUDA(cudaMemcpyAsync(counts, b + o_c, 4 * (size_t)B, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaMemcpyAsync(out, b, 24 * N, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaMemcpyAsync(out_colors, b + o_oc, 24 * N, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaStreamSynchronize(nullptr));
  return PSULVSB_OK;
}

}  // namespace

}  // namespace psulvsb

using psulvsb::fail;

extern "C" {

// ---- voxel downsampling with colours (DESIGN.md section 10, "Voxel downsampling with colours")
unsigned long long psulvsb_voxel_down_sample_colors_workspace_bytes(int n) {
  if (n < 0) return 0ull;
  const psulvsb_fpfh_cloud_t c{nullptr, n, {0.0, 0.0, 0.0}};
  return (unsigned long long)psulvsb::colors_workspace(psulvsb::fpfh_sizes(&c, 1));
}

unsigned long long psulvsb_voxel_down_sample_colors_batch_workspace_bytes(const psulvsb_color_cloud_t* clouds, int B) {
  if (B <= 0 || !clouds) return 0ull;
  for (int c = 0; c < B; ++c)
    if (clouds[c].n < 0) return 0ull;
  const std::vector<psulvsb_fpfh_cloud_t> f = psulvsb::point_clouds(clouds, B);
  return (unsigned long long)psulvsb::colors_workspace(psulvsb::fpfh_sizes(f.data(), B));
}

int psulvsb_voxel_down_sample_colors(void* stream, const double* d_pts, const double* d_colors, int n,
                                     double voxel_size, void* d_work, double* d_out, double* d_out_colors,
                                     int* d_count) {
  if (n < 0 || !psulvsb::voxel_ok(voxel_size) || !d_count ||
      (n > 0 && (!d_pts || !d_colors || !d_work || !d_out || !d_out_colors)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_voxel_down_sample_colors: bad argument (voxel_size must be finite and > 0)");
  const psulvsb_color_cloud_t c{d_pts, n, d_colors, nullptr};
  if (int rc = psulvsb::colors_check(&c, 1, "psulvsb_voxel_down_sample_colors")) return rc;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_voxel_colors((cudaStream_t)stream, &c, 1, voxel_size, d_work, d_out, d_out_colors, d_count);
}

int psulvsb_voxel_down_sample_colors_host(const double* pts, const double* colors, int n, double voxel_size,
                                          double* out, double* out_colors, int* n_out) {
  if (n < 0 || !psulvsb::voxel_ok(voxel_size) || !n_out || (n > 0 && (!pts || !colors || !out || !out_colors)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_voxel_down_sample_colors_host: bad argument (voxel_size must be finite and > 0)");
  *n_out = 0;
  const psulvsb_color_cloud_t c{pts, n, colors, nullptr};
  if (int rc = psulvsb::colors_check(&c, 1, "psulvsb_voxel_down_sample_colors_host")) return rc;
  if (n == 0) return PSULVSB_OK;  // the zero count is written on the host: no device needed
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_voxel_colors_host(&c, 1, voxel_size, out, out_colors, n_out,
                                        "psulvsb_voxel_down_sample_colors_host");
}

int psulvsb_voxel_down_sample_colors_batch(void* stream, const psulvsb_color_cloud_t* clouds, int B,
                                           double voxel_size, void* d_work, double* d_out, double* d_out_colors,
                                           int* d_counts) {
  if (B < 0 || !psulvsb::voxel_ok(voxel_size) || (B > 0 && (!clouds || !d_work || !d_out || !d_out_colors || !d_counts)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_voxel_down_sample_colors_batch: bad argument (voxel_size must be finite and > 0)");
  if (int rc = psulvsb::colors_check(clouds, B, "psulvsb_voxel_down_sample_colors_batch")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_voxel_colors((cudaStream_t)stream, clouds, B, voxel_size, d_work, d_out, d_out_colors, d_counts);
}

int psulvsb_voxel_down_sample_colors_batch_host(const psulvsb_color_cloud_t* clouds, int B, double voxel_size,
                                                double* out, double* out_colors, int* counts) {
  if (B < 0 || !psulvsb::voxel_ok(voxel_size) || (B > 0 && (!clouds || !out || !out_colors || !counts)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_voxel_down_sample_colors_batch_host: bad argument (voxel_size must be finite and > 0)");
  if (int rc = psulvsb::colors_check(clouds, B, "psulvsb_voxel_down_sample_colors_batch_host")) return rc;
  const std::vector<psulvsb_fpfh_cloud_t> f = psulvsb::point_clouds(clouds, B);
  if (psulvsb::fpfh_sizes(f.data(), B).n == 0) {  // zero counts, written on the host: no device needed
    std::memset(counts, 0, sizeof(int) * (size_t)B);
    return PSULVSB_OK;
  }
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_voxel_colors_host(clouds, B, voxel_size, out, out_colors, counts,
                                        "psulvsb_voxel_down_sample_colors_batch_host");
}

}  // extern "C"
