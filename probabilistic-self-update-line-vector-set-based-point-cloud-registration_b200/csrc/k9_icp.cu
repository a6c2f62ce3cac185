// k9_icp.cu -- rigid ICP over two raw clouds, point-to-point (Umeyama without scale) or point-to-plane (Open3D's
// linearisation), in the loop of Open3D's registration_icp: the refinement users of TEASER++ run after the global
// solve.  DESIGN.md section 11 is the specification; oracle/icp.py restates it in numpy.
//
// The target does not move, so its grid is built once per call: cell size h = d (1 + 1e-6), cells floor((x - c) / h)
// in FP64 relative to the target's bounding-box corner c (a pair within d is never two cells apart, also far from the
// origin), hashed into 2^ceil(log2 n_t) buckets (grid.cuh) whose members sit in ascending index order as FP64 records
// (x, y, z, index).  Every round then evaluates the current transform T_k, which lives in device memory:
//   k9_icp_correspond  one thread per source point: transform, nearest target within d over the 27 cells, per-CTA sums;
//   k9_icp_cross       (point-to-point) the centred cross-covariance H over the correspondences, per-CTA sums;
//   k9_icp_step        one CTA: the CTA sums in a fixed order, trace record k, the stop rule, the update U, T <- U T.
// The host issues max_iterations + 1 rounds without looking at the device; once the loop has stopped, the state's
// `done` flag makes every remaining launch return at once.  No floating-point atomics: every result is bit-identical
// from call to call.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "grid.cuh"
#include "svd3.cuh"

namespace psulvsb {

namespace {

constexpr int ICP_THREADS = 128;
constexpr int STEP_THREADS = 1024;
constexpr int STEP_RUNS = STEP_THREADS / 32;
constexpr int NV_P2P = 8;   // count, sum d^2, sum p' (3), sum q (3)
constexpr int NV_P2L = 29;  // count, sum d^2, J^T J (21, upper triangle row by row), J^T r (6)
constexpr int NV_CROSS = 9;  // H, row-major

struct IcpState {
  double R[9];  // row-major
  double t[3];
  double corner[3];  // the target's bounding-box corner: origin of the grid's cells
  double mu_p[3], mu_q[3];
  double fitness, rmse;  // of the last evaluation
  int n_corr;
  int iter;  // updates applied
  int done;
  int status;
};

struct IcpInit {
  double R[9];  // row-major
  double t[3];
};

struct IcpGrid {
  const double4* rec;  // [n in the grid] sorted by bucket, ascending index inside a bucket; .w = index
  const int* start;    // [nb + 1]
  unsigned int mask;   // nb - 1
  double inv_h;
};

__device__ __forceinline__ long long icp_cell(double x, double c, double inv_h) {
  return (long long)floor(dmul(dsub(x, c), inv_h));
}

// ((R00 x + R01 y) + R02 z) + t0, unfused: the restatement evaluates the same expression in numpy
__device__ __forceinline__ void transform_point(const double* R, const double* t, double x, double y, double z,
                                                double& ox, double& oy, double& oz) {
  ox = dadd(dadd(dadd(dmul(R[0], x), dmul(R[1], y)), dmul(R[2], z)), t[0]);
  oy = dadd(dadd(dadd(dmul(R[3], x), dmul(R[4], y)), dmul(R[5], z)), t[1]);
  oz = dadd(dadd(dadd(dmul(R[6], x), dmul(R[7], y)), dmul(R[8], z)), t[2]);
}

// per-CTA sums of c[0, NV): a fixed shuffle tree in each warp, then the warps in order; partials is value-major
template <int NV>
__device__ __forceinline__ void cta_partials(const double (&c)[NV], double* __restrict__ partials) {
  __shared__ double sh[NV][ICP_THREADS / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    double x = c[v];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
    if (lane == 0) sh[v][wid] = x;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s = sh[threadIdx.x][0];
#pragma unroll
    for (int w = 1; w < ICP_THREADS / 32; ++w) s += sh[threadIdx.x][w];
    partials[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = s;
  }
}

// ---- target grid: corner and state, count, (k8_scan, k8_grid_scatter), order
__global__ void __launch_bounds__(STEP_THREADS)
    k9_icp_bounds(const double* __restrict__ tgt, int n, IcpInit init, IcpState* __restrict__ st) {
  __shared__ double red[3][STEP_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  double m[3] = {INFINITY, INFINITY, INFINITY};
  for (int i = tid; i < n; i += STEP_THREADS)
    for (int r = 0; r < 3; ++r) m[r] = fmin(m[r], tgt[3 * (size_t)i + r]);
  for (int r = 0; r < 3; ++r) {
    for (int o = 16; o > 0; o >>= 1) m[r] = fmin(m[r], __shfl_xor_sync(0xffffffffu, m[r], o));
    if (lane == 0) red[r][wid] = m[r];
  }
  __syncthreads();
  if (tid != 0) return;
  for (int r = 0; r < 3; ++r) {
    double c = red[r][0];
    for (int w = 1; w < STEP_THREADS / 32; ++w) c = fmin(c, red[r][w]);
    st->corner[r] = c;
    st->t[r] = init.t[r];
    st->mu_p[r] = st->mu_q[r] = 0.0;
  }
  for (int e = 0; e < 9; ++e) st->R[e] = init.R[e];
  st->fitness = st->rmse = 0.0;
  st->n_corr = st->iter = st->done = st->status = 0;
}

// a target point with a non-finite normal is no candidate of point-to-plane: it stays out of the grid (bucket -1)
__global__ void __launch_bounds__(GRID_THREADS)
    k9_icp_grid_count(const double* __restrict__ tgt, int n, const double* __restrict__ normals,
                      const IcpState* __restrict__ st, double inv_h, unsigned int mask, int* __restrict__ pbucket,
                      int* __restrict__ count) {
  const int i = blockIdx.x * GRID_THREADS + threadIdx.x;
  if (i >= n) return;
  if (normals && !(isfinite(normals[3 * (size_t)i]) && isfinite(normals[3 * (size_t)i + 1]) &&
                   isfinite(normals[3 * (size_t)i + 2]))) {
    pbucket[i] = -1;
    return;
  }
  const double* q = tgt + 3 * (size_t)i;
  const unsigned int b = bucket_of(icp_cell(q[0], st->corner[0], inv_h), icp_cell(q[1], st->corner[1], inv_h),
                                   icp_cell(q[2], st->corner[2], inv_h), mask);
  pbucket[i] = (int)b;
  atomicAdd(count + b, 1);
}

// the scatter's order inside a bucket depends on timing: rank each member by index instead
__global__ void __launch_bounds__(GRID_THREADS)
    k9_icp_grid_order(const double* __restrict__ tgt, int n, const int* __restrict__ pbucket,
                      const int* __restrict__ start, unsigned int nb, const int* __restrict__ tmp,
                      double4* __restrict__ rec) {
  const int p = blockIdx.x * GRID_THREADS + threadIdx.x;
  if (p >= n || p >= start[nb]) return;
  const int i = tmp[p];
  const int b = pbucket[i], s0 = start[b], s1 = start[b + 1];
  int rank = 0;
  for (int q = s0; q < s1; ++q) rank += tmp[q] < i;
  rec[s0 + rank] = make_double4(tgt[3 * (size_t)i], tgt[3 * (size_t)i + 1], tgt[3 * (size_t)i + 2], (double)i);
}

// ---- evaluation of T_k: corr[i] = the target at the smallest d^2 <= dd (ties: lowest index) or -1, and the CTA sums
// of what the step needs (point-to-point: count, sum d^2, sum p', sum q; point-to-plane: count, sum d^2, J^T J, J^T r)
template <bool P2L>
__global__ void __launch_bounds__(ICP_THREADS)
    k9_icp_correspond(IcpGrid g, const double* __restrict__ src, int ns, const double* __restrict__ normals,
                      const IcpState* __restrict__ st, double dd, int* __restrict__ corr,
                      double* __restrict__ partials) {
  if (st->done) return;
  constexpr int NV = P2L ? NV_P2L : NV_P2P;
  const int i = blockIdx.x * ICP_THREADS + threadIdx.x;
  double c[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) c[v] = 0.0;
  if (i < ns) {
    double px, py, pz;
    transform_point(st->R, st->t, src[3 * (size_t)i], src[3 * (size_t)i + 1], src[3 * (size_t)i + 2], px, py, pz);
    const long long cx = icp_cell(px, st->corner[0], g.inv_h), cy = icp_cell(py, st->corner[1], g.inv_h),
                    cz = icp_cell(pz, st->corner[2], g.inv_h);
    // the 27 cells in a fixed order (dz, dy, dx), each bucket once: visit bit k = first cell of its bucket
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
    double best = INFINITY, qx = 0.0, qy = 0.0, qz = 0.0;
    int bj = -1;
#pragma unroll 1
    for (int k = 0; k < 27; ++k) {
      if (!((visit >> k) & 1u)) continue;
      const unsigned int b = bucket_of(cx + k % 3 - 1, cy + (k / 3) % 3 - 1, cz + k / 9 - 1, g.mask);
      const int e = g.start[b + 1];
      for (int u = g.start[b]; u < e; ++u) {
        const double4 q = g.rec[u];
        const double dx = dsub(q.x, px), dy = dsub(q.y, py), dz = dsub(q.z, pz);
        const double d2 = dadd(dadd(dmul(dx, dx), dmul(dy, dy)), dmul(dz, dz));
        const int j = (int)q.w;
        if (d2 <= dd && (d2 < best || (d2 == best && j < bj))) {
          best = d2;
          bj = j;
          qx = q.x;
          qy = q.y;
          qz = q.z;
        }
      }
    }
    corr[i] = bj;
    if (bj >= 0) {
      c[0] = 1.0;
      c[1] = best;
      if constexpr (!P2L) {
        c[2] = px;
        c[3] = py;
        c[4] = pz;
        c[5] = qx;
        c[6] = qy;
        c[7] = qz;
      } else {
        const double nx = normals[3 * (size_t)bj], ny = normals[3 * (size_t)bj + 1], nz = normals[3 * (size_t)bj + 2];
        // r = (p' - q) . n, J = [p' x n, n] (Open3D TransformationEstimationPointToPlane)
        const double r = dadd(dadd(dmul(dsub(px, qx), nx), dmul(dsub(py, qy), ny)), dmul(dsub(pz, qz), nz));
        const double J[6] = {dsub(dmul(py, nz), dmul(pz, ny)), dsub(dmul(pz, nx), dmul(px, nz)),
                             dsub(dmul(px, ny), dmul(py, nx)), nx, ny, nz};
        int v = 2;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
          for (int e = a; e < 6; ++e) c[v++] = dmul(J[a], J[e]);
#pragma unroll
        for (int a = 0; a < 6; ++a) c[23 + a] = dmul(J[a], r);
      }
    }
  }
  cta_partials<NV>(c, partials);
}

// ---- point-to-point: H = sum (p' - mu_p)(q - mu_q)^T over the correspondences of T_k
__global__ void __launch_bounds__(ICP_THREADS)
    k9_icp_cross(const double* __restrict__ src, int ns, const double* __restrict__ tgt, const int* __restrict__ corr,
                 const IcpState* __restrict__ st, double* __restrict__ partials) {
  if (st->done) return;
  const int i = blockIdx.x * ICP_THREADS + threadIdx.x;
  double c[NV_CROSS];
#pragma unroll
  for (int v = 0; v < NV_CROSS; ++v) c[v] = 0.0;
  const int j = i < ns ? corr[i] : -1;
  if (j >= 0) {
    double p[3];
    transform_point(st->R, st->t, src[3 * (size_t)i], src[3 * (size_t)i + 1], src[3 * (size_t)i + 2], p[0], p[1], p[2]);
    double a[3], b[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      a[r] = dsub(p[r], st->mu_p[r]);
      b[r] = dsub(tgt[3 * (size_t)j + r], st->mu_q[r]);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int s = 0; s < 3; ++s) c[3 * r + s] = dmul(a[r], b[s]);
  }
  cta_partials<NV_CROSS>(c, partials);
}

// 6x6 Cholesky of the J^T J upper triangle A (21 entries) and solve A x = -g; false on a non-positive pivot or a
// non-finite solution
__device__ bool solve6(const double* A, const double* g, double x[6]) {
  double L[6][6], y[6];
  int idx[6][6];
  for (int a = 0, v = 0; a < 6; ++a)
    for (int e = a; e < 6; ++e) idx[a][e] = idx[e][a] = v++;
  for (int j = 0; j < 6; ++j) {
    double d = A[idx[j][j]];
    for (int k = 0; k < j; ++k) d -= L[j][k] * L[j][k];
    if (!(d > 0.0)) return false;
    L[j][j] = sqrt(d);
    for (int i = j + 1; i < 6; ++i) {
      double s = A[idx[i][j]];
      for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
      L[i][j] = s / L[j][j];
    }
  }
  for (int i = 0; i < 6; ++i) {
    double s = -g[i];
    for (int k = 0; k < i; ++k) s -= L[i][k] * y[k];
    y[i] = s / L[i][i];
  }
  for (int i = 5; i >= 0; --i) {
    double s = y[i];
    for (int k = i + 1; k < 6; ++k) s -= L[k][i] * x[k];
    x[i] = s / L[i][i];
  }
  for (int i = 0; i < 6; ++i)
    if (!isfinite(x[i])) return false;
  return true;
}

// T <- U T with U = (Ru, tu), Ru row-major
__device__ void compose(IcpState* st, const double Ru[3][3], const double tu[3]) {
  double R[9], t[3];
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) R[3 * r + c] = Ru[r][0] * st->R[c] + Ru[r][1] * st->R[3 + c] + Ru[r][2] * st->R[6 + c];
    t[r] = Ru[r][0] * st->t[0] + Ru[r][1] * st->t[1] + Ru[r][2] * st->t[2] + tu[r];
  }
  for (int e = 0; e < 9; ++e) st->R[e] = R[e];
  for (int r = 0; r < 3; ++r) st->t[r] = t[r];
  st->iter += 1;
}

__device__ void write_transform(const IcpState* st, double* rotation, double* translation) {
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) rotation[3 * c + r] = st->R[3 * r + c];
    translation[r] = st->t[r];
  }
}

struct StepParams {
  int ns, max_iterations;
  double relative_fitness, relative_rmse;
};

// phase 0 (after k9_icp_correspond): record k, stop rule, point-to-plane update or point-to-point means;
// phase 1 (after k9_icp_cross): the point-to-point update
template <bool P2L>
__global__ void __launch_bounds__(STEP_THREADS)
    k9_icp_step(int phase, const double* __restrict__ partials, int nblk, StepParams prm, IcpState* __restrict__ st,
                psulvsb_icp_iteration_t* __restrict__ trace, psulvsb_icp_result_t* __restrict__ result) {
  __shared__ double run[STEP_RUNS][32];
  __shared__ double S[32];
  if (st->done) return;
  const int nv = phase ? NV_CROSS : (P2L ? NV_P2L : NV_P2P);
  // CTA partials: STEP_RUNS contiguous runs summed in index order, then the runs in order
  const int tid = threadIdx.x, v = tid & 31, run_id = tid >> 5;
  const int len = (nblk + STEP_RUNS - 1) / STEP_RUNS, b0 = run_id * len, b1 = min(nblk, b0 + len);
  double s = 0.0;
  if (v < nv)
    for (int b = b0; b < b1; ++b) s += partials[(size_t)v * nblk + b];
  run[run_id][v] = s;
  __syncthreads();
  if (tid < nv) {
    double x = run[0][tid];
    for (int r = 1; r < STEP_RUNS; ++r) x += run[r][tid];
    S[tid] = x;
  }
  __syncthreads();
  if (tid != 0) return;
  if (phase == 1) {
    double H[3][3], Ru[3][3], tu[3];
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) H[r][c] = S[3 * r + c];
    kabsch_rotation(H, Ru);
    for (int r = 0; r < 3; ++r)
      tu[r] = st->mu_q[r] - (Ru[r][0] * st->mu_p[0] + Ru[r][1] * st->mu_p[1] + Ru[r][2] * st->mu_p[2]);
    compose(st, Ru, tu);
    return;
  }
  const int cnt = (int)S[0];
  const double fitness = (double)cnt / (double)prm.ns;
  const double rmse = cnt > 0 ? sqrt(S[1] / (double)cnt) : 0.0;
  const int k = st->iter;
  if (trace) {
    psulvsb_icp_iteration_t* rec = trace + k;
    write_transform(st, rec->rotation, rec->translation);
    rec->fitness = fitness;
    rec->inlier_rmse = rmse;
    rec->n_correspondences = cnt;
  }
  const bool converged = k > 0 && fabs(fitness - st->fitness) < prm.relative_fitness &&
                         fabs(rmse - st->rmse) < prm.relative_rmse;
  st->fitness = fitness;
  st->rmse = rmse;
  st->n_corr = cnt;
  int status = -1;
  if (converged)
    status = PSULVSB_ICP_CONVERGED;
  else if (k >= prm.max_iterations)
    status = PSULVSB_ICP_MAX_ITERATIONS;
  else if (cnt < (P2L ? 6 : 3))
    status = PSULVSB_ICP_NO_UPDATE;
  else if (P2L) {
    double x[6];
    if (!solve6(S + 2, S + 23, x)) {
      status = PSULVSB_ICP_NO_UPDATE;
    } else {
      // U = [Rz(x2) Ry(x1) Rx(x0) | x3..5]
      const double ca = cos(x[0]), sa = sin(x[0]), cb = cos(x[1]), sb = sin(x[1]), cg = cos(x[2]), sg = sin(x[2]);
      const double Ru[3][3] = {{cg * cb, cg * sb * sa - sg * ca, cg * sb * ca + sg * sa},
                               {sg * cb, sg * sb * sa + cg * ca, sg * sb * ca - cg * sa},
                               {-sb, cb * sa, cb * ca}};
      const double tu[3] = {x[3], x[4], x[5]};
      compose(st, Ru, tu);
    }
  } else {
    for (int r = 0; r < 3; ++r) {
      st->mu_p[r] = S[2 + r] / (double)cnt;
      st->mu_q[r] = S[5 + r] / (double)cnt;
    }
  }
  if (status >= 0) {
    st->status = status;
    st->done = 1;
    write_transform(st, result->rotation, result->translation);
    result->fitness = fitness;
    result->inlier_rmse = rmse;
    result->n_correspondences = cnt;
    result->iterations = st->iter;
    result->status = status;
  }
}

inline size_t up256(size_t x) { return (x + 255) & ~size_t(255); }
inline int blocks(long long n, int t) { return (int)((n + t - 1) / t); }

struct IcpWork {
  IcpState* state;
  double4* rec;
  int *pbucket, *count, *start, *cursor, *tmp, *corr;
  double* partials;
};

size_t icp_layout(int ns, int nt, char* base, IcpWork* w) {
  const size_t NS = (size_t)(ns > 0 ? ns : 0), NT = (size_t)(nt > 0 ? nt : 0), nb = bucket_count(nt);
  const size_t nblk = (NS + ICP_THREADS - 1) / ICP_THREADS;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += up256(bytes);
    return p;
  };
  IcpWork v;
  v.state = (IcpState*)take(sizeof(IcpState));
  v.rec = (double4*)take(32 * NT);
  v.pbucket = (int*)take(4 * NT);
  v.count = (int*)take(4 * nb);
  v.start = (int*)take(4 * (nb + 1));
  v.cursor = (int*)take(4 * nb);
  v.tmp = (int*)take(4 * NT);
  v.corr = (int*)take(4 * NS);
  v.partials = (double*)take(8 * (size_t)NV_P2L * nblk);
  if (w) *w = v;
  return off;
}

bool icp_params_ok(const psulvsb_icp_params_t* p) {
  return p && std::isfinite(p->max_correspondence_distance) && p->max_correspondence_distance > 0.0 &&
         p->max_iterations >= 0 && p->relative_fitness >= 0.0 && p->relative_rmse >= 0.0 &&
         (p->point_to_plane == 0 || p->point_to_plane == 1);
}

bool transform_ok(const double* R0, const double* t0) {
  if (!R0 || !t0) return false;
  for (int e = 0; e < 9; ++e)
    if (!std::isfinite(R0[e])) return false;
  for (int r = 0; r < 3; ++r)
    if (!std::isfinite(t0[r])) return false;
  return true;
}

// an empty cloud: T0, fitness 0, no update (one trace record, every correspondence -1)
void empty_result(const double* R0, const double* t0, psulvsb_icp_result_t* res, psulvsb_icp_iteration_t* rec) {
  *res = psulvsb_icp_result_t{};
  *rec = psulvsb_icp_iteration_t{};
  for (int e = 0; e < 9; ++e) res->rotation[e] = rec->rotation[e] = R0[e];
  for (int r = 0; r < 3; ++r) res->translation[r] = rec->translation[r] = t0[r];
  res->status = PSULVSB_ICP_NO_UPDATE;
}

int run_icp(cudaStream_t st, const double* src, int ns, const double* tgt, int nt, const double* normals,
            const psulvsb_icp_params_t& prm, const double* R0, const double* t0, void* work,
            psulvsb_icp_result_t* d_result, psulvsb_icp_iteration_t* d_trace, int* d_corr) {
  IcpWork w;
  icp_layout(ns, nt, static_cast<char*>(work), &w);
  const bool p2l = prm.point_to_plane != 0;
  const double d = prm.max_correspondence_distance;
  const unsigned int nb = bucket_count(nt);
  IcpInit init;
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) init.R[3 * r + c] = R0[3 * c + r];
    init.t[r] = t0[r];
  }
  const IcpGrid g{w.rec, w.start, nb - 1, 1.0 / (d * (1.0 + 1e-6))};
  k9_icp_bounds<<<1, STEP_THREADS, 0, st>>>(tgt, nt, init, w.state);
  PSU_CHECK_LAUNCH("k9_icp_bounds");
  PSU_CUDA(cudaMemsetAsync(w.count, 0, 4 * (size_t)nb, st));
  k9_icp_grid_count<<<blocks(nt, GRID_THREADS), GRID_THREADS, 0, st>>>(tgt, nt, p2l ? normals : nullptr, w.state,
                                                                       g.inv_h, g.mask, w.pbucket, w.count);
  PSU_CHECK_LAUNCH("k9_icp_grid_count");
  k8_scan<<<1, SCAN_THREADS, 0, st>>>(w.count, (int)nb, w.start, w.cursor);
  PSU_CHECK_LAUNCH("k8_scan");
  k8_grid_scatter<<<blocks(nt, GRID_THREADS), GRID_THREADS, 0, st>>>(nt, w.pbucket, w.cursor, w.tmp);
  PSU_CHECK_LAUNCH("k8_grid_scatter");
  k9_icp_grid_order<<<blocks(nt, GRID_THREADS), GRID_THREADS, 0, st>>>(tgt, nt, w.pbucket, w.start, nb, w.tmp, w.rec);
  PSU_CHECK_LAUNCH("k9_icp_grid_order");
  const int nblk = blocks(ns, ICP_THREADS);
  const StepParams sp{ns, prm.max_iterations, prm.relative_fitness, prm.relative_rmse};
  const double dd = d * d;
  for (int k = 0; k <= prm.max_iterations; ++k) {
    if (p2l) {
      k9_icp_correspond<true><<<nblk, ICP_THREADS, 0, st>>>(g, src, ns, normals, w.state, dd, w.corr, w.partials);
      k9_icp_step<true><<<1, STEP_THREADS, 0, st>>>(0, w.partials, nblk, sp, w.state, d_trace, d_result);
    } else {
      k9_icp_correspond<false><<<nblk, ICP_THREADS, 0, st>>>(g, src, ns, nullptr, w.state, dd, w.corr, w.partials);
      k9_icp_step<false><<<1, STEP_THREADS, 0, st>>>(0, w.partials, nblk, sp, w.state, d_trace, d_result);
      if (k < prm.max_iterations) {
        k9_icp_cross<<<nblk, ICP_THREADS, 0, st>>>(src, ns, tgt, w.corr, w.state, w.partials);
        k9_icp_step<false><<<1, STEP_THREADS, 0, st>>>(1, w.partials, nblk, sp, w.state, d_trace, d_result);
      }
    }
    PSU_CHECK_LAUNCH("k9_icp round");
  }
  if (d_corr) PSU_CUDA(cudaMemcpyAsync(d_corr, w.corr, 4 * (size_t)ns, cudaMemcpyDeviceToDevice, st));
  return PSULVSB_OK;
}

}  // namespace

}  // namespace psulvsb

using psulvsb::fail;

extern "C" {

void psulvsb_icp_default_params(psulvsb_icp_params_t* p) {
  if (!p) return;
  p->max_correspondence_distance = 0.0;
  p->relative_fitness = 1e-6;
  p->relative_rmse = 1e-6;
  p->max_iterations = 30;
  p->point_to_plane = 0;
}

unsigned long long psulvsb_icp_workspace_bytes(int n_s, int n_t) {
  return (n_s < 0 || n_t < 0) ? 0ull : (unsigned long long)psulvsb::icp_layout(n_s, n_t, nullptr, nullptr);
}

int psulvsb_icp(void* stream, const double* d_src, int n_s, const double* d_tgt, int n_t, const double* d_tgt_normals,
                const psulvsb_icp_params_t* params, const double R0[9], const double t0[3], void* d_work,
                psulvsb_icp_result_t* d_result, psulvsb_icp_iteration_t* d_trace, int* d_corr) {
  if (n_s < 0 || n_t < 0 || !psulvsb::icp_params_ok(params) || !psulvsb::transform_ok(R0, t0) || !d_result ||
      (params->point_to_plane && !d_tgt_normals) || (n_s > 0 && !d_src) || (n_t > 0 && !d_tgt) ||
      (n_s > 0 && n_t > 0 && !d_work))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_icp: bad argument");
  if (int rc = psulvsb::need_device()) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (n_s == 0 || n_t == 0) {
    psulvsb_icp_result_t res;
    psulvsb_icp_iteration_t rec;
    psulvsb::empty_result(R0, t0, &res, &rec);
    PSU_CUDA(cudaMemcpyAsync(d_result, &res, sizeof res, cudaMemcpyHostToDevice, st));
    if (d_trace) PSU_CUDA(cudaMemcpyAsync(d_trace, &rec, sizeof rec, cudaMemcpyHostToDevice, st));
    if (d_corr && n_s) PSU_CUDA(cudaMemsetAsync(d_corr, 0xFF, 4 * (size_t)n_s, st));
    return PSULVSB_OK;
  }
  return psulvsb::run_icp(st, d_src, n_s, d_tgt, n_t, d_tgt_normals, *params, R0, t0, d_work, d_result, d_trace,
                          d_corr);
}

int psulvsb_icp_host(const double* src, int n_s, const double* tgt, int n_t, const double* tgt_normals,
                     const psulvsb_icp_params_t* params, const double R0[9], const double t0[3],
                     psulvsb_icp_result_t* result, psulvsb_icp_iteration_t* trace, int* corr) {
  if (n_s < 0 || n_t < 0 || !psulvsb::icp_params_ok(params) || !psulvsb::transform_ok(R0, t0) || !result ||
      (params->point_to_plane && !tgt_normals) || (n_s > 0 && !src) || (n_t > 0 && !tgt))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_icp_host: bad argument");
  if (int rc = psulvsb::need_device()) return rc;
  if (n_s == 0 || n_t == 0) {
    psulvsb_icp_iteration_t rec;
    psulvsb::empty_result(R0, t0, result, &rec);
    if (trace) *trace = rec;
    for (int i = 0; corr && i < n_s; ++i) corr[i] = -1;
    return PSULVSB_OK;
  }
  using psulvsb::up256;
  const bool p2l = params->point_to_plane != 0;
  const size_t NS = (size_t)n_s, NT = (size_t)n_t, nrec = (size_t)params->max_iterations + 1;
  // outputs first and contiguous, so that one copy brings them back
  const size_t o_trace = up256(sizeof(psulvsb_icp_result_t)), o_corr = o_trace + sizeof(psulvsb_icp_iteration_t) * nrec,
               o_end = o_corr + 4 * NS, o_src = up256(o_end), o_tgt = o_src + up256(24 * NS),
               o_nrm = o_tgt + up256(24 * NT), o_work = o_nrm + (p2l ? up256(24 * NT) : 0);
  void* buf = nullptr;
  if (cudaMalloc(&buf, o_work + psulvsb_icp_workspace_bytes(n_s, n_t)) != cudaSuccess) {
    cudaGetLastError();
    return fail(PSULVSB_ERR_CUDA, "psulvsb_icp_host: cudaMalloc failed");
  }
  char* b = static_cast<char*>(buf);
  std::vector<char> out(o_end);
  int rc = PSULVSB_OK;
  auto step = [&](cudaError_t e, const char* what) {
    if (!rc && e != cudaSuccess) rc = fail(PSULVSB_ERR_CUDA, std::string("psulvsb_icp_host: ") + what + ": " +
                                                                cudaGetErrorString(e));
  };
  step(cudaMemcpy(b + o_src, src, 24 * NS, cudaMemcpyHostToDevice), "copy in");
  step(cudaMemcpy(b + o_tgt, tgt, 24 * NT, cudaMemcpyHostToDevice), "copy in");
  if (p2l) step(cudaMemcpy(b + o_nrm, tgt_normals, 24 * NT, cudaMemcpyHostToDevice), "copy in");
  if (!rc)
    rc = psulvsb::run_icp(nullptr, (const double*)(b + o_src), n_s, (const double*)(b + o_tgt), n_t,
                          p2l ? (const double*)(b + o_nrm) : nullptr, *params, R0, t0, b + o_work,
                          (psulvsb_icp_result_t*)b, (psulvsb_icp_iteration_t*)(b + o_trace), (int*)(b + o_corr));
  if (!rc) step(cudaMemcpy(out.data(), b, o_end, cudaMemcpyDeviceToHost), "copy out");
  cudaFree(buf);
  if (rc) return rc;
  std::memcpy(result, out.data(), sizeof *result);
  if (trace) std::memcpy(trace, out.data() + o_trace, sizeof(psulvsb_icp_iteration_t) * (size_t)(result->iterations + 1));
  if (corr) std::memcpy(corr, out.data() + o_corr, 4 * NS);
  return PSULVSB_OK;
}

}  // extern "C"
