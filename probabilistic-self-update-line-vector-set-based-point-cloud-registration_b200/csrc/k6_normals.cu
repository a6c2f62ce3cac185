// k6_normals.cu -- surface normals by k-nearest-neighbour PCA: what the reference driver obtains from PCL
// before its timed region (examples/teaser_cpp_ply/PSULVSB.cc:35-85: pcl::NormalEstimation, setKSearch(20),
// default viewpoint (0, 0, 0)) and feeds to the normal-angle histogram pre-filter.
//
// One thread per query point: all points stream through shared memory in FP32 tiles; the thread keeps its
// k best (squared distance, index) pairs sorted in local memory (the query itself is its own nearest
// neighbour, as with PCL's nearestKSearch on the same cloud); then mean + covariance of the k neighbours in
// FP64, the eigenvector of the smallest eigenvalue by cyclic Jacobi, flipped towards the viewpoint
// (pcl::flipNormalTowardsViewpoint).  O(n^2) distance evaluations: 1.3e9 for the full 36k-vertex bunny.
// PCL's own eigen-solver and tie handling are not pinned by the reference -> parity unpinned; the tests
// compare with a numpy restatement (oracle/prefilter.py).
#include <cuda_runtime.h>

#include "common.cuh"
#include "engine.cuh"
#include "eig3.cuh"

namespace psulvsb {

namespace {

constexpr int NRM_THREADS = 128;
constexpr int NRM_TILE = 1024;
constexpr int NRM_KMAX = 32;

__global__ void __launch_bounds__(NRM_THREADS)
    knn_normals_kernel(const double* __restrict__ pts, int n, int k, double vx, double vy, double vz,
                       double* __restrict__ normals) {
  __shared__ float4 tile[NRM_TILE];
  const int i = blockIdx.x * NRM_THREADS + threadIdx.x;
  const bool live = i < n;
  float qx = 0.f, qy = 0.f, qz = 0.f;
  if (live) {
    qx = (float)pts[3 * (size_t)i];
    qy = (float)pts[3 * (size_t)i + 1];
    qz = (float)pts[3 * (size_t)i + 2];
  }
  float bd[NRM_KMAX];
  int bi[NRM_KMAX];
  for (int t = 0; t < k; ++t) {
    bd[t] = 3.0e38f;
    bi[t] = -1;
  }
  for (int j0 = 0; j0 < n; j0 += NRM_TILE) {
    __syncthreads();
    for (int t = threadIdx.x; t < NRM_TILE; t += NRM_THREADS) {
      const int j = j0 + t;
      tile[t] = j < n ? make_float4((float)pts[3 * (size_t)j], (float)pts[3 * (size_t)j + 1],
                                    (float)pts[3 * (size_t)j + 2], 0.f)
                      : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();
    if (!live) continue;
    const int lim = min(NRM_TILE, n - j0);
    for (int t = 0; t < lim; ++t) {
      const float dx = tile[t].x - qx, dy = tile[t].y - qy, dz = tile[t].z - qz;
      const float d = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
      if (d < bd[k - 1]) {  // insertion into the sorted list (ties keep the lower index first)
        int pos = k - 1;
        while (pos > 0 && bd[pos - 1] > d) {
          bd[pos] = bd[pos - 1];
          bi[pos] = bi[pos - 1];
          --pos;
        }
        bd[pos] = d;
        bi[pos] = j0 + t;
      }
    }
  }
  if (!live) return;
  // mean and covariance of the neighbourhood (FP64, from the original coordinates)
  double mean[3] = {0, 0, 0};
  int cnt = 0;
  for (int t = 0; t < k; ++t)
    if (bi[t] >= 0) {
      for (int r = 0; r < 3; ++r) mean[r] += pts[3 * (size_t)bi[t] + r];
      ++cnt;
    }
  if (cnt < 3) {  // PCL answers NaN for a neighbourhood that cannot define a plane
    for (int r = 0; r < 3; ++r) normals[3 * (size_t)i + r] = nan("");
    return;
  }
  for (int r = 0; r < 3; ++r) mean[r] /= (double)cnt;
  double cov[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
  for (int t = 0; t < k; ++t)
    if (bi[t] >= 0) {
      double d[3];
      for (int r = 0; r < 3; ++r) d[r] = pts[3 * (size_t)bi[t] + r] - mean[r];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) cov[r][c] += d[r] * d[c];
    }
  double nv[3];
  smallest_eigenvector(cov, nv);
  const double px = pts[3 * (size_t)i], py = pts[3 * (size_t)i + 1], pz = pts[3 * (size_t)i + 2];
  if ((vx - px) * nv[0] + (vy - py) * nv[1] + (vz - pz) * nv[2] < 0.0) {  // flipNormalTowardsViewpoint
    nv[0] = -nv[0];
    nv[1] = -nv[1];
    nv[2] = -nv[2];
  }
  for (int r = 0; r < 3; ++r) normals[3 * (size_t)i + r] = nv[r];
}

}  // namespace

int launch_knn_normals(cudaStream_t st, const double* pts, int n, int k, const double* viewpoint, double* normals) {
  if (n <= 0) return PSULVSB_OK;
  if (k < 3 || k > NRM_KMAX) return fail(PSULVSB_ERR_INVALID, "knn normals: k must be in [3, 32]");
  const double vx = viewpoint ? viewpoint[0] : 0.0, vy = viewpoint ? viewpoint[1] : 0.0, vz = viewpoint ? viewpoint[2] : 0.0;
  knn_normals_kernel<<<(n + NRM_THREADS - 1) / NRM_THREADS, NRM_THREADS, 0, st>>>(pts, n, k, vx, vy, vz, normals);
  PSU_CHECK_LAUNCH("knn_normals_kernel");
  return PSULVSB_OK;
}

}  // namespace psulvsb
