// k8_colors.cu -- the colour gradients of colored ICP (Open3D's InitializePointCloudForColoredICP) on FPFH's grid:
// per point, the least-squares gradient of the intensity over its hybrid neighbourhood in the tangent plane.  DESIGN.md
// section 11 ("Colored ICP") is the specification; tests/colored_icp_restatement.py restates it in numpy.  Colored ICP
// (k9_icp.cu) runs this stage on its targets through run_color_gradients.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "ft_batch.cuh"
#include "ft_grid.cuh"
#include "grid.cuh"

namespace psulvsb {

namespace {

// ---- colour gradients (DESIGN.md section 11, "Colored ICP"; Open3D's InitializePointCloudForColoredICP).  A cloud's
// colours and normals travel in a side table of the batch, indexed by cloud.
struct ColorSide {
  const double* colors;   // 3 x n
  const double* normals;  // 3 x n
};

// A g = b for the symmetric A = (A00, A01, A02, A11, A12, A22) by Cholesky, every operation in the order written
// (tests/colored_icp_restatement.py repeats it); false on a non-positive pivot or a non-finite g
__device__ __forceinline__ bool solve3(const double A[6], const double b[3], double g[3]) {
  if (!(A[0] > 0.0)) return false;
  const double L00 = __dsqrt_rn(A[0]);
  const double L10 = __ddiv_rn(A[1], L00), L20 = __ddiv_rn(A[2], L00);
  const double d1 = dsub(A[3], dmul(L10, L10));
  if (!(d1 > 0.0)) return false;
  const double L11 = __dsqrt_rn(d1);
  const double L21 = __ddiv_rn(dsub(A[4], dmul(L20, L10)), L11);
  const double d2 = dsub(dsub(A[5], dmul(L20, L20)), dmul(L21, L21));
  if (!(d2 > 0.0)) return false;
  const double L22 = __dsqrt_rn(d2);
  const double y0 = __ddiv_rn(b[0], L00);
  const double y1 = __ddiv_rn(dsub(b[1], dmul(L10, y0)), L11);
  const double y2 = __ddiv_rn(dsub(dsub(b[2], dmul(L20, y0)), dmul(L21, y1)), L22);
  g[2] = __ddiv_rn(y2, L22);
  g[1] = __ddiv_rn(dsub(y1, dmul(L21, g[2])), L11);
  g[0] = __ddiv_rn(dsub(dsub(y0, dmul(L10, g[1])), dmul(L20, g[2])), L00);
  return isfinite(g[0]) && isfinite(g[1]) && isfinite(g[2]);
}

// one thread per sorted point of a batch of clouds: the hybrid neighbourhood (hybrid_threshold, the point itself
// counted), nn kept points; nn >= 4 and a finite normal n: every kept j != i adds the row a = (q_j - ((q_j - q_i).n) n)
// - q_i, b = I_j - I_i to A^T A and A^T b in the walk's order, the row (nn - 1) n (b = 0) comes last, and g solves the
// 3x3 system; otherwise, or when the solve fails, g = 0
__global__ void __launch_bounds__(FT_THREADS)
    k8_color_gradients(const FtCloud* __restrict__ clouds, const ColorSide* __restrict__ side,
                       const int* __restrict__ tile_first, int B, double inv_h, const float4* __restrict__ spts,
                       const int* __restrict__ start, float r2, int max_nn, double* __restrict__ gradients) {
  const int ci = pair_of(tile_first, B, blockIdx.x);
  const FtCloud& cl = clouds[ci];
  const int p = (blockIdx.x - tile_first[ci]) * FT_THREADS + threadIdx.x;
  if (p >= cl.n) return;
  const Grid g{inv_h, cl.mask, spts, start + cl.b0 + ci};
  const float4 me = spts[cl.p0 + p];
  const int i = __float_as_int(me.w);
  __shared__ unsigned long long kept[FT_MAX_NN][FT_THREADS];
  const Hybrid hy = hybrid_threshold<true>(g, me, r2, max_nn, kept, threadIdx.x);
  const unsigned long long kstar = hy.kstar;
  const int nk = hy.nk;
  const int nn = min(nk, max_nn);
  const double *pts = cl.pts, *col = side[ci].colors, *nrm = side[ci].normals;
  const double nx = nrm[3 * (size_t)i], ny = nrm[3 * (size_t)i + 1], nz = nrm[3 * (size_t)i + 2];
  double gv[3] = {0.0, 0.0, 0.0};
  if (nn >= 4 && isfinite(nx) && isfinite(ny) && isfinite(nz)) {
    const double qx = pts[3 * (size_t)i], qy = pts[3 * (size_t)i + 1], qz = pts[3 * (size_t)i + 2];
    const double Ii = intensity(col + 3 * (size_t)i);
    double A[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, b[3] = {0.0, 0.0, 0.0};
    for_neighbours_masked(g, me, r2, [&](float4 q, int j) {
      if (j == i || nn_key(me, q, j) > kstar) return;
      const double* v = pts + 3 * (size_t)j;
      const double s = dadd(dadd(dmul(dsub(v[0], qx), nx), dmul(dsub(v[1], qy), ny)), dmul(dsub(v[2], qz), nz));
      const double a[3] = {dsub(dsub(v[0], dmul(s, nx)), qx), dsub(dsub(v[1], dmul(s, ny)), qy),
                           dsub(dsub(v[2], dmul(s, nz)), qz)};
      const double bj = dsub(intensity(col + 3 * (size_t)j), Ii);
#pragma unroll
      for (int r = 0, e = 0; r < 3; ++r) {
#pragma unroll
        for (int c = r; c < 3; ++c, ++e) A[e] = dadd(A[e], dmul(a[r], a[c]));
        b[r] = dadd(b[r], dmul(a[r], bj));
      }
    });
    const double w = (double)(nn - 1);
    const double c[3] = {dmul(w, nx), dmul(w, ny), dmul(w, nz)};
#pragma unroll
    for (int r = 0, e = 0; r < 3; ++r)
#pragma unroll
      for (int cc = r; cc < 3; ++cc, ++e) A[e] = dadd(A[e], dmul(c[r], c[cc]));
    double x[3];
    if (solve3(A, b, x))
      for (int r = 0; r < 3; ++r) gv[r] = x[r];
  }
  const size_t o = (size_t)cl.p0 + i;
  for (int r = 0; r < 3; ++r) gradients[3 * o + r] = gv[r];
}

// ---- colour gradients on the host side: FPFH's grid of cell size `radius` over the clouds' points, then
// k8_color_gradients.  A batch always takes the batched grid kernels, so cloud c's gradients are those of a batch of
// cloud c alone.
std::vector<psulvsb_fpfh_cloud_t> grid_clouds(const psulvsb_color_cloud_t* clouds, int B) {
  std::vector<psulvsb_fpfh_cloud_t> f((size_t)B);
  for (int c = 0; c < B; ++c) f[c] = psulvsb_fpfh_cloud_t{clouds[c].points, clouds[c].n, {0.0, 0.0, 0.0}};
  return f;
}

struct ColorWork {
  FtCloud* cloud;  // [B], followed by tile_first [B + 1]: one copy uploads both (cloud_table)
  int* tile_first;
  size_t table_bytes;
  ColorSide* side;                     // [B]
  float4* spts;                        // [n] sorted by bucket, ascending index inside a bucket
  int *pbucket, *tmp;                  // [n]
  int *count, *cursor;                 // [nb]
  int* start;                          // [nb + B]
};

size_t color_layout(const FpfhSizes& z, char* base, ColorWork* w) {
  const size_t nn = (size_t)z.n, nb = (size_t)z.nb, B = (size_t)z.B;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += up256(bytes);
    return p;
  };
  ColorWork v;
  v.table_bytes = sizeof(FtCloud) * B + 4 * (B + 1);
  v.cloud = (FtCloud*)take(v.table_bytes);
  v.tile_first = (int*)((char*)v.cloud + sizeof(FtCloud) * B);
  v.side = (ColorSide*)take(sizeof(ColorSide) * B);
  v.spts = (float4*)take(16 * nn);
  v.pbucket = (int*)take(4 * nn);
  v.tmp = (int*)take(4 * nn);
  v.count = (int*)take(4 * nb);
  v.cursor = (int*)take(4 * nb);
  v.start = (int*)take(4 * (nb + B));
  if (w) *w = v;
  return off;
}

// PSULVSB_ERR_INVALID for a bad cloud, PSULVSB_ERR_UNSUPPORTED for concatenations past the int range, else OK
int color_clouds_check(const psulvsb_color_cloud_t* clouds, int B, const char* who) {
  for (int c = 0; c < B; ++c)
    if (clouds[c].n > 0 && (!clouds[c].colors || !clouds[c].normals))
      return fail(PSULVSB_ERR_INVALID, std::string(who) + ": bad cloud " + std::to_string(c));
  const std::vector<psulvsb_fpfh_cloud_t> f = grid_clouds(clouds, B);
  return clouds_check(f.data(), B, who);
}

bool gradient_args_ok(double radius, int max_nn) {
  return std::isfinite(radius) && radius > 0.0 && max_nn >= 4 && max_nn <= FT_MAX_NN;
}

// the batch on host buffers (clouds checked, B >= 1): points, colours and normals go up in one copy, the gradients
// come back in one
int run_color_gradients_host(const psulvsb_color_cloud_t* clouds, int B, double radius, int max_nn, double* gradients,
                             const char* who) {
  const std::vector<psulvsb_fpfh_cloud_t> f = grid_clouds(clouds, B);
  const FpfhSizes z = fpfh_sizes(f.data(), B);
  if (z.n == 0) return PSULVSB_OK;
  const size_t N = (size_t)z.n, o_in = up256(24 * N), o_w = o_in + up256(3 * 24 * N);
  std::vector<char> in(3 * 24 * N);
  std::vector<psulvsb_color_cloud_t> dev(clouds, clouds + B);
  DevBuf buf;
  if (int rc = buf.alloc(o_w + color_gradients_scratch(clouds, B), who)) return rc;
  char* b = static_cast<char*>(buf.p);
  size_t off = 0;
  for (int c = 0; c < B; ++c) {
    if (dev[c].n <= 0) continue;
    const size_t bytes = 24 * (size_t)dev[c].n;
    const double** arrays[3] = {&dev[c].points, &dev[c].colors, &dev[c].normals};
    for (const double** a : arrays) {
      std::memcpy(in.data() + off, *a, bytes);
      *a = reinterpret_cast<const double*>(b + o_in + off);
      off += bytes;
    }
  }
  PSU_CUDA(cudaMemcpyAsync(b + o_in, in.data(), in.size(), cudaMemcpyHostToDevice, nullptr));
  if (int rc = run_color_gradients(nullptr, dev.data(), B, radius, max_nn, b + o_w, (double*)b)) return rc;
  PSU_CUDA(cudaMemcpyAsync(gradients, b, 24 * N, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaStreamSynchronize(nullptr));
  return PSULVSB_OK;
}

}  // namespace

size_t color_gradients_scratch(const psulvsb_color_cloud_t* clouds, int B) {
  const std::vector<psulvsb_fpfh_cloud_t> f = grid_clouds(clouds, B);
  return color_layout(fpfh_sizes(f.data(), B), nullptr, nullptr);
}

int run_color_gradients(cudaStream_t st, const psulvsb_color_cloud_t* clouds, int B, double radius, int max_nn,
                        void* work, double* gradients) {
  const std::vector<psulvsb_fpfh_cloud_t> f = grid_clouds(clouds, B);
  const FpfhSizes z = fpfh_sizes(f.data(), B);
  if (z.tiles == 0) return PSULVSB_OK;
  ColorWork w;
  color_layout(z, static_cast<char*>(work), &w);
  const std::vector<char> table = cloud_table(f.data(), B, w.table_bytes);
  std::vector<ColorSide> side((size_t)B);
  for (int c = 0; c < B; ++c) side[c] = ColorSide{clouds[c].colors, clouds[c].normals};
  PSU_CUDA(cudaMemcpyAsync(w.cloud, table.data(), table.size(), cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaMemcpyAsync(w.side, side.data(), sizeof(ColorSide) * (size_t)B, cudaMemcpyHostToDevice, st));
  const double inv_h = 1.0 / (radius * (1.0 + 1e-5));
  const float r2 = (float)(radius * radius);
  const int tiles = (int)z.tiles, n = (int)z.n;
  const FtCloud& one = *reinterpret_cast<const FtCloud*>(table.data());  // unused by the batched kernels
  PSU_CUDA(cudaMemsetAsync(w.count, 0, 4 * (size_t)z.nb, st));
  k8_grid_count<true><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, inv_h, w.pbucket, w.count);
  k8_cloud_scan<true><<<B, SCAN_THREADS, 0, st>>>(w.cloud, one, w.count, w.start, w.cursor);
  k8_grid_scatter<<<blocks(n, GRID_THREADS), GRID_THREADS, 0, st>>>(n, w.pbucket, w.cursor, w.tmp);
  k8_grid_order<true><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, w.pbucket, w.start, w.tmp, w.spts);
  k8_color_gradients<<<tiles, FT_THREADS, 0, st>>>(w.cloud, w.side, w.tile_first, B, inv_h, w.spts, w.start, r2, max_nn,
                                                   gradients);
  PSU_CHECK_LAUNCH("k8_color_gradients");
  return PSULVSB_OK;
}

}  // namespace psulvsb

using psulvsb::fail;

extern "C" {

// ---- colour gradients alone (DESIGN.md section 11, "Colored ICP")
unsigned long long psulvsb_color_gradients_batch_workspace_bytes(const psulvsb_color_cloud_t* clouds, int B) {
  if (B <= 0 || !clouds) return 0ull;
  for (int c = 0; c < B; ++c)
    if (clouds[c].n < 0) return 0ull;
  return (unsigned long long)psulvsb::color_gradients_scratch(clouds, B);
}

int psulvsb_color_gradients_batch(void* stream, const psulvsb_color_cloud_t* clouds, int B, double radius, int max_nn,
                                  void* d_work, double* d_gradients) {
  if (B < 0 || !psulvsb::gradient_args_ok(radius, max_nn) || (B > 0 && (!clouds || !d_work || !d_gradients)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_color_gradients_batch: bad argument (radius finite and > 0, max_nn 4..32)");
  if (int rc = psulvsb::color_clouds_check(clouds, B, "psulvsb_color_gradients_batch")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_color_gradients((cudaStream_t)stream, clouds, B, radius, max_nn, d_work, d_gradients);
}

int psulvsb_color_gradients_batch_host(const psulvsb_color_cloud_t* clouds, int B, double radius, int max_nn,
                                       double* gradients) {
  if (B < 0 || !psulvsb::gradient_args_ok(radius, max_nn) || (B > 0 && (!clouds || !gradients)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_color_gradients_batch_host: bad argument (radius finite and > 0, max_nn 4..32)");
  if (int rc = psulvsb::color_clouds_check(clouds, B, "psulvsb_color_gradients_batch_host")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_color_gradients_host(clouds, B, radius, max_nn, gradients, "psulvsb_color_gradients_batch_host");
}

}  // extern "C"
