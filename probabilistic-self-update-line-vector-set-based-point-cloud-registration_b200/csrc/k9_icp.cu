// k9_icp.cu -- rigid ICP over two raw clouds, point-to-point (Umeyama without scale), point-to-plane (Open3D's
// linearisation) or generalized ICP (plane-to-plane, Segal et al.; Open3D's registration_generalized_icp), in the loop
// of Open3D's registration_icp: the refinement users of TEASER++ run after the global solve.  DESIGN.md section 11 is
// the specification; oracle/icp.py restates ICP in numpy, tests/gicp_restatement.py generalized ICP.
//
// A call refines a batch of B independent pairs that share the parameters (one pair for psulvsb_icp); every launch
// covers all of them.  Each pair's target does not move, so its grid is built once per call: cell size h = d (1 + 1e-6),
// cells floor((x - c) / h) in FP64 relative to the target's bounding-box corner c (a pair within d is never two cells
// apart, also far from the origin), hashed into the pair's own table of 2^ceil(log2 n_t) buckets (grid.cuh) whose
// members sit in ascending index order as FP64 records (x, y, z, index).  Every round then evaluates each pair's
// current transform T_k, which lives in device memory:
//   k9_icp_correspond  one thread per source point, one CTA per (pair, 128-point tile): transform, nearest target
//                      within d over the 27 cells, per-CTA sums (point-to-plane: the 6x6 system's terms);
//   k9_gicp_correspond the same pass for generalized ICP, whose per-CTA sums are its 6x6 system's terms;
//   k9_icp_cross       (point-to-point) the centred cross-covariance H over the correspondences, per-CTA sums;
//   k9_icp_step        one CTA per pair: the pair's CTA sums in a fixed order, trace record k, the stop rule, the
//                      update U, T <- U T.
// A CTA finds its pair by a binary search over the prefix of the pairs' tile counts.  Tiles, bucket tables and the
// order of every sum depend on the pair's own sizes only, so a pair's results are bit-identical whatever else is in the
// batch.  The host issues max_iterations + 1 rounds without looking at the device; once a pair's loop has stopped, its
// state's `done` flag makes its CTAs of every remaining launch return at once.  No floating-point atomics: every result
// is bit-identical from call to call.
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
constexpr int NV_P2L = 29;  // count, sum d^2, J^T J (21, upper triangle row by row), J^T r (6); GICP's A^T M A, A^T M d
constexpr int NV_CROSS = 9;  // H, row-major

// the objective of a call: the correspondence and step kernels are instantiated per mode
enum Mode : int { P2P = 0, P2L = 1, GICP = 2 };

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

// one pair on the device: the caller's pair and where the pair sits in the batch's concatenations
struct IcpPair {
  const double* src;
  const double* tgt;
  const double* nrm;   // target normals: point-to-plane and GICP, else nullptr
  const double* snrm;  // source normals: GICP only, else nullptr
  int b0;              // first bucket of the pair's table (count, cursor); its start table begins at b0 + pair
  int ns, nt;          // the caller's sizes
  int s0;              // first source point (correspondences)
  int t0;              // first target point in the grid's arrays (an empty pair has none)
  unsigned int mask;   // nb - 1
  IcpInit init;
  // an empty pair's result is T0 (k9_icp_bounds)
  __host__ __device__ bool live() const { return ns > 0 && nt > 0; }
};
// the pair table is part of the workspace, whose size psulvsb_icp_[batch_]workspace_bytes publish
static_assert(sizeof(IcpPair) == 152, "IcpPair's size fixes the published workspace sizes");

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

// per-CTA sums of c[0, NV) of tile `tile` of a pair with `ntiles` tiles: a fixed shuffle tree in each warp, then the
// warps in order; the pair's partials are value-major
template <int NV>
__device__ __forceinline__ void cta_partials(const double (&c)[NV], double* __restrict__ partials, int ntiles,
                                             int tile) {
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
    partials[(size_t)threadIdx.x * ntiles + tile] = s;
  }
}

__device__ void write_transform(const IcpState* st, double* rotation, double* translation) {
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) rotation[3 * c + r] = st->R[3 * r + c];
    translation[r] = st->t[r];
  }
}

// ---- target grids: corner and state, count, (segmented scan, k8_grid_scatter), order
// one CTA per pair; an empty pair gets its result here: T0, fitness 0, no update, one trace record, every
// correspondence -1
__global__ void __launch_bounds__(STEP_THREADS)
    k9_icp_bounds(const IcpPair* __restrict__ pairs, IcpState* __restrict__ states, int nrec, int* __restrict__ corr,
                  psulvsb_icp_iteration_t* __restrict__ trace, psulvsb_icp_result_t* __restrict__ results) {
  __shared__ double red[3][STEP_THREADS / 32];
  const IcpPair& pr = pairs[blockIdx.x];
  IcpState* st = states + blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n = pr.live() ? pr.nt : 0;
  if (!pr.live())
    for (int i = tid; i < pr.ns; i += STEP_THREADS) corr[pr.s0 + i] = -1;
  double m[3] = {INFINITY, INFINITY, INFINITY};
  for (int i = tid; i < n; i += STEP_THREADS)
    for (int r = 0; r < 3; ++r) m[r] = fmin(m[r], pr.tgt[3 * (size_t)i + r]);
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
    st->t[r] = pr.init.t[r];
    st->mu_p[r] = st->mu_q[r] = 0.0;
  }
  for (int e = 0; e < 9; ++e) st->R[e] = pr.init.R[e];
  st->fitness = st->rmse = 0.0;
  st->n_corr = st->iter = st->done = st->status = 0;
  if (pr.live()) return;
  st->done = 1;
  st->status = PSULVSB_ICP_NO_UPDATE;
  psulvsb_icp_result_t* res = results + blockIdx.x;
  write_transform(st, res->rotation, res->translation);
  res->fitness = res->inlier_rmse = 0.0;
  res->n_correspondences = res->iterations = 0;
  res->status = PSULVSB_ICP_NO_UPDATE;
  if (trace) {
    psulvsb_icp_iteration_t* rec = trace + (size_t)blockIdx.x * nrec;
    write_transform(st, rec->rotation, rec->translation);
    rec->fitness = rec->inlier_rmse = 0.0;
    rec->n_correspondences = 0;
  }
}

// one thread per target point of a live pair (tgt_first: prefix of the pairs' binned targets); with drop_nonfinite
// (point-to-plane) a target point with a non-finite normal is no candidate: it stays out of the grid (bucket -1).
// pbucket holds the bucket's index in the batch's concatenated tables.
__global__ void __launch_bounds__(GRID_THREADS)
    k9_icp_grid_count(const IcpPair* __restrict__ pairs, const int* __restrict__ tgt_first, int B, int n,
                      const IcpState* __restrict__ states, double inv_h, int drop_nonfinite, int* __restrict__ pbucket,
                      int* __restrict__ count) {
  const int i = blockIdx.x * GRID_THREADS + threadIdx.x;
  if (i >= n) return;
  const int p = pair_of(tgt_first, B, i);
  const IcpPair& pr = pairs[p];
  const double* normals = pr.nrm;
  const size_t l = (size_t)(i - pr.t0);
  if (drop_nonfinite && !(isfinite(normals[3 * l]) && isfinite(normals[3 * l + 1]) && isfinite(normals[3 * l + 2]))) {
    pbucket[i] = -1;
    return;
  }
  const double* q = pr.tgt + 3 * l;
  const IcpState* st = states + p;
  const long long b = pr.b0 + bucket_of(icp_cell(q[0], st->corner[0], inv_h), icp_cell(q[1], st->corner[1], inv_h),
                                        icp_cell(q[2], st->corner[2], inv_h), pr.mask);
  pbucket[i] = (int)b;
  atomicAdd(count + b, 1);
}

// one CTA per pair: its bucket table, positions counted from its first target point
__global__ void __launch_bounds__(SCAN_THREADS)
    k9_icp_grid_scan(const IcpPair* __restrict__ pairs, const int* __restrict__ count, int* __restrict__ start,
                     int* __restrict__ cursor) {
  const IcpPair& pr = pairs[blockIdx.x];
  if (!pr.live()) return;
  cta_scan(count + pr.b0, (int)(pr.mask + 1), start + pr.b0 + blockIdx.x, cursor + pr.b0, pr.t0);
}

// one thread per scatter slot; the scatter's order inside a bucket depends on timing: rank each member by index instead
__global__ void __launch_bounds__(GRID_THREADS)
    k9_icp_grid_order(const IcpPair* __restrict__ pairs, const int* __restrict__ tgt_first, int B, int n,
                      const int* __restrict__ pbucket, const int* __restrict__ start, const int* __restrict__ tmp,
                      double4* __restrict__ rec) {
  const int s = blockIdx.x * GRID_THREADS + threadIdx.x;
  if (s >= n) return;
  const int p = pair_of(tgt_first, B, s);
  const IcpPair& pr = pairs[p];
  const int* pstart = start + p;  // the pair's table: pstart[pr.b0, pr.b0 + nb]
  if (s >= pstart[pr.b0 + pr.mask + 1]) return;  // slots of targets left out of the grid
  const int i = tmp[s];
  const int b = pbucket[i], s0 = pstart[b], s1 = pstart[b + 1];
  int rank = 0;
  for (int q = s0; q < s1; ++q) rank += tmp[q] < i;
  const size_t l = (size_t)(i - pr.t0);
  rec[s0 + rank] = make_double4(pr.tgt[3 * l], pr.tgt[3 * l + 1], pr.tgt[3 * l + 2], (double)(i - pr.t0));
}

// ---- generalized ICP's terms of one correspondence (DESIGN.md section 11, "Generalized ICP"); every product and sum
// in the order written, which tests/gicp_restatement.py repeats elementwise in numpy

// n / |n| in FP64, |n| = sqrt((x x + y y) + z z); 0 when that squared length is not finite and positive (a NaN radius
// normal, a zero normal): the point's covariance is then I
__device__ __forceinline__ void unit_normal(const double* n, double u[3]) {
  const double x = n[0], y = n[1], z = n[2];
  const double s2 = dadd(dadd(dmul(x, x), dmul(y, y)), dmul(z, z));
  if (!(isfinite(s2) && s2 > 0.0)) {
    u[0] = u[1] = u[2] = 0.0;
    return;
  }
  const double s = __dsqrt_rn(s2);
  u[0] = __ddiv_rn(x, s);
  u[1] = __ddiv_rn(y, s);
  u[2] = __ddiv_rn(z, s);
}

// a x b = (a1 b2 - a2 b1, a2 b0 - a0 b2, a0 b1 - a1 b0)
__device__ __forceinline__ void cross3(const double a[3], double b0, double b1, double b2, double o[3]) {
  o[0] = dsub(dmul(a[1], b2), dmul(a[2], b1));
  o[1] = dsub(dmul(a[2], b0), dmul(a[0], b2));
  o[2] = dsub(dmul(a[0], b1), dmul(a[1], b0));
}

// c[0, 27): H = A^T M A (upper triangle row by row) and g = A^T M d for A = [-[p']x, I3], d = p' - q,
// M = C^-1, C = Sigma_t + R Sigma_s R^T = 2 I - w (m m^T + n n^T) with m = R n_s-hat, n = n_t-hat (0 for a side whose
// covariance is I, which drops its term exactly), w = 1 - epsilon.  With S = -[p']x (S^T x = p' x x) and K = M S
// (row r: p' x M_r): H = [[S^T K, K^T], [K, M]], g = [p' x (M d), M d].
__device__ __forceinline__ void gicp_terms(const double p[3], const double q[3], const double m[3], const double n[3],
                                           double w, double* __restrict__ c) {
  const double C00 = dsub(2.0, dmul(w, dadd(dmul(m[0], m[0]), dmul(n[0], n[0]))));
  const double C01 = dsub(0.0, dmul(w, dadd(dmul(m[0], m[1]), dmul(n[0], n[1]))));
  const double C02 = dsub(0.0, dmul(w, dadd(dmul(m[0], m[2]), dmul(n[0], n[2]))));
  const double C11 = dsub(2.0, dmul(w, dadd(dmul(m[1], m[1]), dmul(n[1], n[1]))));
  const double C12 = dsub(0.0, dmul(w, dadd(dmul(m[1], m[2]), dmul(n[1], n[2]))));
  const double C22 = dsub(2.0, dmul(w, dadd(dmul(m[2], m[2]), dmul(n[2], n[2]))));
  // M = adj(C) / det(C); det(C) >= 8 epsilon^3 > 0
  const double A00 = dsub(dmul(C11, C22), dmul(C12, C12)), A01 = dsub(dmul(C02, C12), dmul(C01, C22)),
               A02 = dsub(dmul(C01, C12), dmul(C02, C11)), A11 = dsub(dmul(C00, C22), dmul(C02, C02)),
               A12 = dsub(dmul(C01, C02), dmul(C00, C12)), A22 = dsub(dmul(C00, C11), dmul(C01, C01));
  const double det = dadd(dadd(dmul(C00, A00), dmul(C01, A01)), dmul(C02, A02));
  const double M00 = __ddiv_rn(A00, det), M01 = __ddiv_rn(A01, det), M02 = __ddiv_rn(A02, det),
               M11 = __ddiv_rn(A11, det), M12 = __ddiv_rn(A12, det), M22 = __ddiv_rn(A22, det);
  const double Mr[3][3] = {{M00, M01, M02}, {M01, M11, M12}, {M02, M12, M22}};
  const double d[3] = {dsub(p[0], q[0]), dsub(p[1], q[1]), dsub(p[2], q[2])};
  double e[3];  // M d
#pragma unroll
  for (int r = 0; r < 3; ++r) e[r] = dadd(dadd(dmul(Mr[r][0], d[0]), dmul(Mr[r][1], d[1])), dmul(Mr[r][2], d[2]));
  double K[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r) cross3(p, Mr[r][0], Mr[r][1], Mr[r][2], K[r]);
  double SK[3][3];  // S^T K, column b = p' x (column b of K)
#pragma unroll
  for (int b = 0; b < 3; ++b) {
    double o[3];
    cross3(p, K[0][b], K[1][b], K[2][b], o);
#pragma unroll
    for (int a = 0; a < 3; ++a) SK[a][b] = o[a];
  }
  int v = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int b = a; b < 3; ++b) c[v++] = SK[a][b];
#pragma unroll
    for (int b = 0; b < 3; ++b) c[v++] = K[b][a];
  }
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = a; b < 3; ++b) c[v++] = Mr[a][b];
  double pe[3];
  cross3(p, e[0], e[1], e[2], pe);
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    c[21 + a] = pe[a];
    c[24 + a] = e[a];
  }
}

// ---- evaluation of T_k: corr[i] = the target at the smallest d^2 <= dd (ties: lowest index) or -1, and the CTA sums
// of what the step needs (point-to-point: count, sum d^2, sum p', sum q; point-to-plane: count, sum d^2, J^T J, J^T r;
// GICP: count, sum d^2, A^T M A, A^T M d with w = 1 - epsilon); the body of k9_icp_correspond and k9_gicp_correspond
template <int MODE>
__device__ __forceinline__ void correspond(const IcpPair* __restrict__ pairs, const int* __restrict__ tile_first, int B,
                                           const double4* __restrict__ rec, const int* __restrict__ start,
                                           double inv_h, const IcpState* __restrict__ states, double dd, double w,
                                           int* __restrict__ corr, double* __restrict__ partials) {
  // the pair, its bucket mask and its start table are read from shared memory at each use: held in registers across
  // the 27-cell walk they push the point-to-plane instantiation past 128 registers (4 CTAs per SM) into spills
  __shared__ volatile int s_pair, s_start;
  __shared__ volatile unsigned int s_mask;
  const int p = pair_of(tile_first, B, blockIdx.x);
  const IcpState* st = states + p;
  if (st->done) return;
  if (threadIdx.x == 0) {
    s_pair = p;
    s_start = (int)(pairs[p].b0 + p);
    s_mask = pairs[p].mask;
  }
  __syncthreads();
  constexpr int NV = MODE == P2P ? NV_P2P : NV_P2L;
  const int i = (blockIdx.x - tile_first[p]) * ICP_THREADS + threadIdx.x;
  double c[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) c[v] = 0.0;
  if (i < pairs[p].ns) {
    const double* src = pairs[p].src;
    double px, py, pz;
    transform_point(st->R, st->t, src[3 * (size_t)i], src[3 * (size_t)i + 1], src[3 * (size_t)i + 2], px, py, pz);
    const long long cx = icp_cell(px, st->corner[0], inv_h), cy = icp_cell(py, st->corner[1], inv_h),
                    cz = icp_cell(pz, st->corner[2], inv_h);
    // the 27 cells in a fixed order (dz, dy, dx), each bucket once: visit bit k = first cell of its bucket
    unsigned int visit = 0;
    {
      unsigned int b[27];
#pragma unroll
      for (int k = 0; k < 27; ++k) {
        b[k] = bucket_of(cx + k % 3 - 1, cy + (k / 3) % 3 - 1, cz + k / 9 - 1, s_mask);
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
      const unsigned int b = bucket_of(cx + k % 3 - 1, cy + (k / 3) % 3 - 1, cz + k / 9 - 1, s_mask);
      const int e = start[s_start + b + 1];
      for (int u = start[s_start + b]; u < e; ++u) {
        const double4 q = rec[u];
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
    corr[pairs[s_pair].s0 + i] = bj;
    if (bj >= 0) {
      c[0] = 1.0;
      c[1] = best;
      if constexpr (MODE == P2P) {
        c[2] = px;
        c[3] = py;
        c[4] = pz;
        c[5] = qx;
        c[6] = qy;
        c[7] = qz;
      } else if constexpr (MODE == P2L) {
        const double* normals = pairs[s_pair].nrm;
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
      } else {
        // the walk is done: only now are the normals read, m = R_k n_s-hat in transform_point's order
        double a[3], n[3], m[3];
        unit_normal(pairs[s_pair].snrm + 3 * (size_t)i, a);
        unit_normal(pairs[s_pair].nrm + 3 * (size_t)bj, n);
        const double* R = st->R;
#pragma unroll
        for (int r = 0; r < 3; ++r) m[r] = dadd(dadd(dmul(R[3 * r], a[0]), dmul(R[3 * r + 1], a[1])), dmul(R[3 * r + 2], a[2]));
        const double pp[3] = {px, py, pz}, qq[3] = {qx, qy, qz};
        gicp_terms(pp, qq, m, n, w, c + 2);
      }
    }
  }
  const int tile0 = tile_first[s_pair];
  cta_partials<NV>(c, partials + (size_t)NV_P2L * tile0, tile_first[s_pair + 1] - tile0, blockIdx.x - tile0);
}

// point-to-point (MODE P2P) and point-to-plane (P2L)
template <int MODE>
__global__ void __launch_bounds__(ICP_THREADS)
    k9_icp_correspond(const IcpPair* __restrict__ pairs, const int* __restrict__ tile_first, int B,
                      const double4* __restrict__ rec, const int* __restrict__ start, double inv_h,
                      const IcpState* __restrict__ states, double dd, int* __restrict__ corr,
                      double* __restrict__ partials) {
  correspond<MODE>(pairs, tile_first, B, rec, start, inv_h, states, dd, 0.0, corr, partials);
}

// generalized ICP, w = 1 - epsilon: the same pass under its own name
__global__ void __launch_bounds__(ICP_THREADS)
    k9_gicp_correspond(const IcpPair* __restrict__ pairs, const int* __restrict__ tile_first, int B,
                       const double4* __restrict__ rec, const int* __restrict__ start, double inv_h,
                       const IcpState* __restrict__ states, double dd, double w, int* __restrict__ corr,
                       double* __restrict__ partials) {
  correspond<GICP>(pairs, tile_first, B, rec, start, inv_h, states, dd, w, corr, partials);
}

// ---- point-to-point: H = sum (p' - mu_p)(q - mu_q)^T over the correspondences of T_k
__global__ void __launch_bounds__(ICP_THREADS)
    k9_icp_cross(const IcpPair* __restrict__ pairs, const int* __restrict__ tile_first, int B,
                 const int* __restrict__ corr, const IcpState* __restrict__ states, double* __restrict__ partials) {
  const int p = pair_of(tile_first, B, blockIdx.x);
  const IcpState* st = states + p;
  if (st->done) return;
  const IcpPair& pr = pairs[p];
  const int tile0 = tile_first[p], tile = blockIdx.x - tile0;
  const int i = tile * ICP_THREADS + threadIdx.x;
  double c[NV_CROSS];
#pragma unroll
  for (int v = 0; v < NV_CROSS; ++v) c[v] = 0.0;
  const int j = i < pr.ns ? corr[pr.s0 + i] : -1;
  if (j >= 0) {
    const double *src = pr.src, *tgt = pr.tgt;
    double p3[3];
    transform_point(st->R, st->t, src[3 * (size_t)i], src[3 * (size_t)i + 1], src[3 * (size_t)i + 2], p3[0], p3[1],
                    p3[2]);
    double a[3], b[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      a[r] = dsub(p3[r], st->mu_p[r]);
      b[r] = dsub(tgt[3 * (size_t)j + r], st->mu_q[r]);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int s = 0; s < 3; ++s) c[3 * r + s] = dmul(a[r], b[s]);
  }
  cta_partials<NV_CROSS>(c, partials + (size_t)NV_P2L * tile0, tile_first[p + 1] - tile0, tile);
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

struct StepParams {
  int max_iterations;
  double relative_fitness, relative_rmse;
};

// one CTA per pair; phase 0 (after k9_icp_correspond): record k, stop rule, point-to-plane / GICP update or
// point-to-point means; phase 1 (after k9_icp_cross): the point-to-point update
template <int MODE>
__global__ void __launch_bounds__(STEP_THREADS)
    k9_icp_step(int phase, const IcpPair* __restrict__ pairs, const int* __restrict__ tile_first,
                const double* __restrict__ partials, StepParams prm, IcpState* __restrict__ states,
                psulvsb_icp_iteration_t* __restrict__ trace, psulvsb_icp_result_t* __restrict__ results) {
  __shared__ double run[STEP_RUNS][32];
  __shared__ double S[32];
  const int p = blockIdx.x;
  IcpState* st = states + p;
  if (st->done) return;
  const int nv = phase ? NV_CROSS : (MODE == P2P ? NV_P2P : NV_P2L);
  const int tile0 = tile_first[p], nblk = tile_first[p + 1] - tile0;
  partials += (size_t)NV_P2L * tile0;
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
  const double fitness = (double)cnt / (double)pairs[p].ns;
  const double rmse = cnt > 0 ? sqrt(S[1] / (double)cnt) : 0.0;
  const int k = st->iter;
  if (trace) {
    psulvsb_icp_iteration_t* rec = trace + (size_t)p * (prm.max_iterations + 1) + k;
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
  else if (cnt < (MODE == P2L ? 6 : 3))
    status = PSULVSB_ICP_NO_UPDATE;
  else if (MODE != P2P) {
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
    psulvsb_icp_result_t* result = results + p;
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

bool live(const psulvsb_icp_pair_t& p) { return p.n_s > 0 && p.n_t > 0; }

// what a batch's workspace depends on: B, the source points of all pairs, and the targets, buckets and 128-point
// source tiles of the pairs that are not empty
struct IcpSizes {
  long long ns = 0, nt = 0, nb = 0, tiles = 0;
  int B = 0;
};

IcpSizes icp_sizes(const psulvsb_icp_pair_t* pairs, int B) {
  IcpSizes z;
  z.B = B;
  for (int b = 0; b < B; ++b) {
    z.ns += pairs[b].n_s;
    if (!live(pairs[b])) continue;
    z.nt += pairs[b].n_t;
    z.nb += bucket_count(pairs[b].n_t);
    z.tiles += (pairs[b].n_s + ICP_THREADS - 1) / ICP_THREADS;
  }
  return z;
}

struct IcpWork {
  IcpPair* pair;                 // [B], followed by tile_first and tgt_first: one copy uploads the three
  int *tile_first, *tgt_first;   // [B + 1] each: prefix of the pairs' tiles, of their binned targets
  IcpState* state;               // [B]
  double4* rec;                  // [nt]
  int *pbucket, *tmp;            // [nt]
  int *count, *cursor;           // [nb]
  int* start;                    // [nb + B]: pair p's table at b0 + p, nb_p + 1 entries
  int* corr;                     // [ns]
  double* partials;              // [NV_P2L * tiles]: pair p's at NV_P2L * tile_first[p], value-major
  size_t table_bytes;            // pair + tile_first + tgt_first
};

size_t icp_layout(const IcpSizes& z, char* base, IcpWork* w) {
  const size_t B = (size_t)z.B;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += up256(bytes);
    return p;
  };
  IcpWork v;
  v.table_bytes = sizeof(IcpPair) * B + 2 * 4 * (B + 1);
  v.pair = (IcpPair*)take(v.table_bytes);
  v.tile_first = (int*)((char*)v.pair + sizeof(IcpPair) * B);
  v.tgt_first = v.tile_first + (B + 1);
  v.state = (IcpState*)take(sizeof(IcpState) * B);
  v.rec = (double4*)take(32 * (size_t)z.nt);
  v.pbucket = (int*)take(4 * (size_t)z.nt);
  v.tmp = (int*)take(4 * (size_t)z.nt);
  v.count = (int*)take(4 * (size_t)z.nb);
  v.cursor = (int*)take(4 * (size_t)z.nb);
  v.start = (int*)take(4 * ((size_t)z.nb + B));
  v.corr = (int*)take(4 * (size_t)z.ns);
  v.partials = (double*)take(8 * (size_t)NV_P2L * (size_t)z.tiles);
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

// PSULVSB_ERR_INVALID for a bad pair, PSULVSB_ERR_UNSUPPORTED for concatenations past the int range, else OK
int pairs_check(const psulvsb_icp_pair_t* pairs, int B, const psulvsb_icp_params_t* params, const char* who) {
  long long ns = 0, nt = 0;
  for (int b = 0; b < B; ++b) {
    const psulvsb_icp_pair_t& p = pairs[b];
    if (p.n_s < 0 || p.n_t < 0 || (p.n_s > 0 && !p.src) || (p.n_t > 0 && !p.tgt) || !transform_ok(p.R0, p.t0) ||
        (params->point_to_plane && p.n_t > 0 && !p.tgt_normals))
      return fail(PSULVSB_ERR_INVALID, std::string(who) + ": bad pair " + std::to_string(b));
    ns += p.n_s;
    nt += p.n_t;
  }
  const IcpSizes z = icp_sizes(pairs, B);
  // the buckets' start tables are indexed by int
  if (ns >= (1ll << 31) || nt >= (1ll << 31) || z.nb + B >= (1ll << 31))
    return fail(PSULVSB_ERR_UNSUPPORTED, std::string(who) + ": the batch's clouds exceed 2^31 - 1 points in all");
  return PSULVSB_OK;
}

// an empty cloud: T0, fitness 0, no update (one trace record, every correspondence -1)
void empty_result(const double* R0, const double* t0, psulvsb_icp_result_t* res, psulvsb_icp_iteration_t* rec) {
  *res = psulvsb_icp_result_t{};
  *rec = psulvsb_icp_iteration_t{};
  for (int e = 0; e < 9; ++e) res->rotation[e] = rec->rotation[e] = R0[e];
  for (int r = 0; r < 3; ++r) res->translation[r] = rec->translation[r] = t0[r];
  res->status = PSULVSB_ICP_NO_UPDATE;
}

// what a call minimises: the mode, GICP's source normals (one pointer per pair, else nullptr) and w = 1 - epsilon
struct Objective {
  Mode mode;
  const double* const* src_normals;
  double w;
};

Objective icp_objective(const psulvsb_icp_params_t& prm) {
  return Objective{prm.point_to_plane ? P2L : P2P, nullptr, 0.0};
}

// the batch on the device (pairs checked, B >= 1): one upload of the pair table, the grids, max_iterations + 1 rounds
// and one copy of the correspondences; the launch count does not depend on B
int run_icp(cudaStream_t st, const psulvsb_icp_pair_t* pairs, int B, const psulvsb_icp_params_t& prm, Objective obj,
            void* work, psulvsb_icp_result_t* d_results, psulvsb_icp_iteration_t* d_trace, int* d_corr) {
  const IcpSizes z = icp_sizes(pairs, B);
  IcpWork w;
  icp_layout(z, static_cast<char*>(work), &w);
  const double d = prm.max_correspondence_distance;
  std::vector<char> table(w.table_bytes);
  IcpPair* hp = reinterpret_cast<IcpPair*>(table.data());
  int* tile_first = reinterpret_cast<int*>(table.data() + sizeof(IcpPair) * (size_t)B);
  int* tgt_first = tile_first + (B + 1);
  long long b0 = 0;
  int s0 = 0;
  tile_first[0] = tgt_first[0] = 0;
  for (int b = 0; b < B; ++b) {
    const psulvsb_icp_pair_t& q = pairs[b];
    IcpPair& h = hp[b];
    h = IcpPair{};
    h.src = q.src;
    h.tgt = q.tgt;
    h.nrm = obj.mode != P2P ? q.tgt_normals : nullptr;
    h.snrm = obj.mode == GICP ? obj.src_normals[b] : nullptr;
    h.ns = q.n_s;
    h.nt = q.n_t;
    h.s0 = s0;
    h.t0 = tgt_first[b];
    h.b0 = (int)b0;
    const unsigned int nb = h.live() ? bucket_count(q.n_t) : 0u;
    h.mask = nb - 1;
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) h.init.R[3 * r + c] = q.R0[3 * c + r];
      h.init.t[r] = q.t0[r];
    }
    s0 += q.n_s;
    b0 += nb;
    tile_first[b + 1] = tile_first[b] + (h.live() ? blocks(q.n_s, ICP_THREADS) : 0);
    tgt_first[b + 1] = tgt_first[b] + (h.live() ? q.n_t : 0);
  }
  PSU_CUDA(cudaMemcpyAsync(w.pair, table.data(), table.size(), cudaMemcpyHostToDevice, st));
  const int nrec = prm.max_iterations + 1;
  k9_icp_bounds<<<B, STEP_THREADS, 0, st>>>(w.pair, w.state, nrec, w.corr, d_trace, d_results);
  PSU_CHECK_LAUNCH("k9_icp_bounds");
  const int nt = (int)z.nt, tiles = (int)z.tiles;
  if (tiles > 0) {
    const double inv_h = 1.0 / (d * (1.0 + 1e-6));
    PSU_CUDA(cudaMemsetAsync(w.count, 0, 4 * (size_t)z.nb, st));
    k9_icp_grid_count<<<blocks(nt, GRID_THREADS), GRID_THREADS, 0, st>>>(w.pair, w.tgt_first, B, nt, w.state, inv_h,
                                                                         obj.mode == P2L, w.pbucket, w.count);
    PSU_CHECK_LAUNCH("k9_icp_grid_count");
    k9_icp_grid_scan<<<B, SCAN_THREADS, 0, st>>>(w.pair, w.count, w.start, w.cursor);
    PSU_CHECK_LAUNCH("k9_icp_grid_scan");
    k8_grid_scatter<<<blocks(nt, GRID_THREADS), GRID_THREADS, 0, st>>>(nt, w.pbucket, w.cursor, w.tmp);
    PSU_CHECK_LAUNCH("k8_grid_scatter");
    k9_icp_grid_order<<<blocks(nt, GRID_THREADS), GRID_THREADS, 0, st>>>(w.pair, w.tgt_first, B, nt, w.pbucket,
                                                                         w.start, w.tmp, w.rec);
    PSU_CHECK_LAUNCH("k9_icp_grid_order");
    const StepParams sp{prm.max_iterations, prm.relative_fitness, prm.relative_rmse};
    const double dd = d * d;
    for (int k = 0; k <= prm.max_iterations; ++k) {
      if (obj.mode == P2L) {
        k9_icp_correspond<P2L><<<tiles, ICP_THREADS, 0, st>>>(w.pair, w.tile_first, B, w.rec, w.start, inv_h,
                                                              w.state, dd, w.corr, w.partials);
        k9_icp_step<P2L><<<B, STEP_THREADS, 0, st>>>(0, w.pair, w.tile_first, w.partials, sp, w.state, d_trace,
                                                     d_results);
      } else if (obj.mode == GICP) {
        k9_gicp_correspond<<<tiles, ICP_THREADS, 0, st>>>(w.pair, w.tile_first, B, w.rec, w.start, inv_h, w.state,
                                                          dd, obj.w, w.corr, w.partials);
        k9_icp_step<GICP><<<B, STEP_THREADS, 0, st>>>(0, w.pair, w.tile_first, w.partials, sp, w.state, d_trace,
                                                      d_results);
      } else {
        k9_icp_correspond<P2P><<<tiles, ICP_THREADS, 0, st>>>(w.pair, w.tile_first, B, w.rec, w.start, inv_h,
                                                              w.state, dd, w.corr, w.partials);
        k9_icp_step<P2P><<<B, STEP_THREADS, 0, st>>>(0, w.pair, w.tile_first, w.partials, sp, w.state, d_trace,
                                                     d_results);
        if (k < prm.max_iterations) {
          k9_icp_cross<<<tiles, ICP_THREADS, 0, st>>>(w.pair, w.tile_first, B, w.corr, w.state, w.partials);
          k9_icp_step<P2P><<<B, STEP_THREADS, 0, st>>>(1, w.pair, w.tile_first, w.partials, sp, w.state, d_trace,
                                                       d_results);
        }
      }
      PSU_CHECK_LAUNCH("k9_icp round");
    }
  }
  if (d_corr && z.ns > 0)
    PSU_CUDA(cudaMemcpyAsync(d_corr, w.corr, 4 * (size_t)z.ns, cudaMemcpyDeviceToDevice, st));
  return PSULVSB_OK;
}

// the batch on host buffers (pairs checked, B >= 1): the live pairs' clouds and normals go up in one copy, results,
// trace records and correspondences come back in one
int run_icp_host(const psulvsb_icp_pair_t* pairs, int B, const psulvsb_icp_params_t& prm, Objective obj,
                 psulvsb_icp_result_t* results, psulvsb_icp_iteration_t* trace, int* corr, const char* who) {
  const bool tn = obj.mode != P2P, sn = obj.mode == GICP;
  const IcpSizes z = icp_sizes(pairs, B);
  const size_t nrec = (size_t)prm.max_iterations + 1, NB = (size_t)B;
  // outputs first and contiguous, so that one copy brings them back
  const size_t o_trace = up256(sizeof(psulvsb_icp_result_t) * NB),
               o_corr = o_trace + (trace ? sizeof(psulvsb_icp_iteration_t) * nrec * NB : 0),
               o_end = o_corr + (corr ? 4 * (size_t)z.ns : 0), o_in = up256(o_end);
  const size_t in_bytes = 24 * (size_t)(z.ns * (sn ? 2 : 1) + z.nt * (tn ? 2 : 1));
  const size_t o_work = up256(o_in + in_bytes);
  // the live pairs' src, tgt (and target normals, then source normals) in pair order: pair b's src at in_off[b], the
  // rest after it
  std::vector<char> in(in_bytes);
  std::vector<size_t> in_off(NB);
  size_t off = 0;
  for (int b = 0; b < B; ++b) {
    const psulvsb_icp_pair_t& q = pairs[b];
    in_off[b] = off;
    if (!live(q)) continue;
    auto put = [&](const double* h, int n) {
      std::memcpy(in.data() + off, h, 24 * (size_t)n);
      off += 24 * (size_t)n;
    };
    put(q.src, q.n_s);
    put(q.tgt, q.n_t);
    if (tn) put(q.tgt_normals, q.n_t);
    if (sn) put(obj.src_normals[b], q.n_s);
  }
  void* buf = nullptr;
  if (cudaMalloc(&buf, o_work + icp_layout(z, nullptr, nullptr)) != cudaSuccess) {
    cudaGetLastError();
    return fail(PSULVSB_ERR_CUDA, std::string(who) + ": cudaMalloc failed");
  }
  char* base = static_cast<char*>(buf);
  std::vector<psulvsb_icp_pair_t> dev(pairs, pairs + B);
  std::vector<const double*> dev_snrm(NB, nullptr);
  for (int b = 0; b < B; ++b) {
    psulvsb_icp_pair_t& q = dev[b];
    const double* src = reinterpret_cast<const double*>(base + o_in + in_off[b]);
    const bool on = live(q);
    q.src = on ? src : nullptr;
    q.tgt = on ? src + 3 * (size_t)q.n_s : nullptr;
    q.tgt_normals = on && tn ? src + 3 * ((size_t)q.n_s + q.n_t) : nullptr;
    dev_snrm[b] = on && sn ? src + 3 * ((size_t)q.n_s + 2 * (size_t)q.n_t) : nullptr;
  }
  Objective dev_obj = obj;
  dev_obj.src_normals = dev_snrm.data();
  std::vector<char> out(o_end);
  int rc = PSULVSB_OK;
  auto step = [&](cudaError_t e, const char* what) {
    if (!rc && e != cudaSuccess)
      rc = fail(PSULVSB_ERR_CUDA, std::string(who) + ": " + what + ": " + cudaGetErrorString(e));
  };
  if (in_bytes) step(cudaMemcpy(base + o_in, in.data(), in_bytes, cudaMemcpyHostToDevice), "copy in");
  if (!rc)
    rc = run_icp(nullptr, dev.data(), B, prm, dev_obj, base + o_work, (psulvsb_icp_result_t*)base,
                 trace ? (psulvsb_icp_iteration_t*)(base + o_trace) : nullptr, corr ? (int*)(base + o_corr) : nullptr);
  if (!rc) step(cudaMemcpy(out.data(), base, o_end, cudaMemcpyDeviceToHost), "copy out");
  cudaFree(buf);
  if (rc) return rc;
  std::memcpy(results, out.data(), sizeof(psulvsb_icp_result_t) * NB);
  for (int b = 0; trace && b < B; ++b)
    std::memcpy(trace + nrec * b, out.data() + o_trace + sizeof(psulvsb_icp_iteration_t) * nrec * b,
                sizeof(psulvsb_icp_iteration_t) * (size_t)(results[b].iterations + 1));
  if (corr) std::memcpy(corr, out.data() + o_corr, 4 * (size_t)z.ns);
  return PSULVSB_OK;
}

// an empty cloud of a single call, without device work: T0, fitness 0, no update, one trace record, corr -1
int empty_device(cudaStream_t st, int n_s, const double* R0, const double* t0, psulvsb_icp_result_t* d_result,
                 psulvsb_icp_iteration_t* d_trace, int* d_corr) {
  psulvsb_icp_result_t res;
  psulvsb_icp_iteration_t rec;
  empty_result(R0, t0, &res, &rec);
  PSU_CUDA(cudaMemcpyAsync(d_result, &res, sizeof res, cudaMemcpyHostToDevice, st));
  if (d_trace) PSU_CUDA(cudaMemcpyAsync(d_trace, &rec, sizeof rec, cudaMemcpyHostToDevice, st));
  if (d_corr && n_s) PSU_CUDA(cudaMemsetAsync(d_corr, 0xFF, 4 * (size_t)n_s, st));
  return PSULVSB_OK;
}

void empty_host(int n_s, const double* R0, const double* t0, psulvsb_icp_result_t* result,
                psulvsb_icp_iteration_t* trace, int* corr) {
  psulvsb_icp_iteration_t rec;
  empty_result(R0, t0, result, &rec);
  if (trace) *trace = rec;
  for (int i = 0; corr && i < n_s; ++i) corr[i] = -1;
}

bool epsilon_ok(double eps) { return std::isfinite(eps) && eps > 0.0 && eps <= 1.0; }

// GICP takes ICP's parameters in point-to-point form: the entry point is the mode
bool gicp_params_ok(const psulvsb_icp_params_t* p, double eps) {
  return icp_params_ok(p) && p->point_to_plane == 0 && epsilon_ok(eps);
}

// GICP pairs as ICP pairs (target normals included) and their source normals; PSULVSB_ERR_INVALID for a pair with both
// clouds non-empty and a normal array missing, else pairs_check's verdict
int gicp_pairs(const psulvsb_gicp_pair_t* g, int B, const psulvsb_icp_params_t* params,
               std::vector<psulvsb_icp_pair_t>& pairs, std::vector<const double*>& src_normals, const char* who) {
  pairs.resize((size_t)B);
  src_normals.resize((size_t)B);
  for (int b = 0; b < B; ++b) {
    const psulvsb_gicp_pair_t& q = g[b];
    if (q.n_s > 0 && q.n_t > 0 && (!q.src_normals || !q.tgt_normals))
      return fail(PSULVSB_ERR_INVALID, std::string(who) + ": bad pair " + std::to_string(b) + " (normals)");
    psulvsb_icp_pair_t& p = pairs[b];
    p.src = q.src;
    p.n_s = q.n_s;
    p.tgt = q.tgt;
    p.n_t = q.n_t;
    p.tgt_normals = q.tgt_normals;
    std::memcpy(p.R0, q.R0, sizeof p.R0);
    std::memcpy(p.t0, q.t0, sizeof p.t0);
    src_normals[b] = q.src_normals;
  }
  return pairs_check(pairs.data(), B, params, who);
}

psulvsb_icp_pair_t one_pair(const double* src, int n_s, const double* tgt, int n_t, const double* normals,
                            const double* R0, const double* t0) {
  psulvsb_icp_pair_t p{};
  p.src = src;
  p.n_s = n_s;
  p.tgt = tgt;
  p.n_t = n_t;
  p.tgt_normals = normals;
  std::memcpy(p.R0, R0, sizeof p.R0);
  std::memcpy(p.t0, t0, sizeof p.t0);
  return p;
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
  if (n_s < 0 || n_t < 0) return 0ull;
  const psulvsb_icp_pair_t p{nullptr, n_s, nullptr, n_t, nullptr, {}, {}};
  return (unsigned long long)psulvsb::icp_layout(psulvsb::icp_sizes(&p, 1), nullptr, nullptr);
}

unsigned long long psulvsb_icp_batch_workspace_bytes(const psulvsb_icp_pair_t* pairs, int B) {
  if (B <= 0 || !pairs) return 0ull;
  for (int b = 0; b < B; ++b)
    if (pairs[b].n_s < 0 || pairs[b].n_t < 0) return 0ull;
  return (unsigned long long)psulvsb::icp_layout(psulvsb::icp_sizes(pairs, B), nullptr, nullptr);
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
  if (n_s == 0 || n_t == 0) return psulvsb::empty_device(st, n_s, R0, t0, d_result, d_trace, d_corr);
  const psulvsb_icp_pair_t p = psulvsb::one_pair(d_src, n_s, d_tgt, n_t, d_tgt_normals, R0, t0);
  return psulvsb::run_icp(st, &p, 1, *params, psulvsb::icp_objective(*params), d_work, d_result, d_trace, d_corr);
}

int psulvsb_icp_host(const double* src, int n_s, const double* tgt, int n_t, const double* tgt_normals,
                     const psulvsb_icp_params_t* params, const double R0[9], const double t0[3],
                     psulvsb_icp_result_t* result, psulvsb_icp_iteration_t* trace, int* corr) {
  if (n_s < 0 || n_t < 0 || !psulvsb::icp_params_ok(params) || !psulvsb::transform_ok(R0, t0) || !result ||
      (params->point_to_plane && !tgt_normals) || (n_s > 0 && !src) || (n_t > 0 && !tgt))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_icp_host: bad argument");
  if (int rc = psulvsb::need_device()) return rc;
  if (n_s == 0 || n_t == 0) {
    psulvsb::empty_host(n_s, R0, t0, result, trace, corr);
    return PSULVSB_OK;
  }
  const psulvsb_icp_pair_t p = psulvsb::one_pair(src, n_s, tgt, n_t, tgt_normals, R0, t0);
  return psulvsb::run_icp_host(&p, 1, *params, psulvsb::icp_objective(*params), result, trace, corr,
                               "psulvsb_icp_host");
}

int psulvsb_icp_batch(void* stream, const psulvsb_icp_pair_t* pairs, int B, const psulvsb_icp_params_t* params,
                      void* d_work, psulvsb_icp_result_t* d_results, psulvsb_icp_iteration_t* d_trace, int* d_corr) {
  if (B < 0 || !psulvsb::icp_params_ok(params) || (B > 0 && (!pairs || !d_work || !d_results)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_icp_batch: bad argument");
  if (int rc = psulvsb::pairs_check(pairs, B, params, "psulvsb_icp_batch")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_icp((cudaStream_t)stream, pairs, B, *params, psulvsb::icp_objective(*params), d_work, d_results,
                          d_trace, d_corr);
}

int psulvsb_icp_batch_host(const psulvsb_icp_pair_t* pairs, int B, const psulvsb_icp_params_t* params,
                           psulvsb_icp_result_t* results, psulvsb_icp_iteration_t* trace, int* corr) {
  if (B < 0 || !psulvsb::icp_params_ok(params) || (B > 0 && (!pairs || !results)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_icp_batch_host: bad argument");
  if (int rc = psulvsb::pairs_check(pairs, B, params, "psulvsb_icp_batch_host")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_icp_host(pairs, B, *params, psulvsb::icp_objective(*params), results, trace, corr,
                               "psulvsb_icp_batch_host");
}

int psulvsb_gicp(void* stream, const double* d_src, int n_s, const double* d_src_normals, const double* d_tgt, int n_t,
                 const double* d_tgt_normals, const psulvsb_icp_params_t* params, double epsilon, const double R0[9],
                 const double t0[3], void* d_work, psulvsb_icp_result_t* d_result, psulvsb_icp_iteration_t* d_trace,
                 int* d_corr) {
  const bool both = n_s > 0 && n_t > 0;
  if (n_s < 0 || n_t < 0 || !psulvsb::gicp_params_ok(params, epsilon) || !psulvsb::transform_ok(R0, t0) ||
      !d_result || (n_s > 0 && !d_src) || (n_t > 0 && !d_tgt) ||
      (both && (!d_work || !d_src_normals || !d_tgt_normals)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_gicp: bad argument");
  if (int rc = psulvsb::need_device()) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (!both) return psulvsb::empty_device(st, n_s, R0, t0, d_result, d_trace, d_corr);
  const psulvsb_icp_pair_t p = psulvsb::one_pair(d_src, n_s, d_tgt, n_t, d_tgt_normals, R0, t0);
  const psulvsb::Objective obj{psulvsb::GICP, &d_src_normals, 1.0 - epsilon};
  return psulvsb::run_icp(st, &p, 1, *params, obj, d_work, d_result, d_trace, d_corr);
}

int psulvsb_gicp_host(const double* src, int n_s, const double* src_normals, const double* tgt, int n_t,
                      const double* tgt_normals, const psulvsb_icp_params_t* params, double epsilon,
                      const double R0[9], const double t0[3], psulvsb_icp_result_t* result,
                      psulvsb_icp_iteration_t* trace, int* corr) {
  const bool both = n_s > 0 && n_t > 0;
  if (n_s < 0 || n_t < 0 || !psulvsb::gicp_params_ok(params, epsilon) || !psulvsb::transform_ok(R0, t0) || !result ||
      (n_s > 0 && !src) || (n_t > 0 && !tgt) || (both && (!src_normals || !tgt_normals)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_gicp_host: bad argument");
  if (int rc = psulvsb::need_device()) return rc;
  if (!both) {
    psulvsb::empty_host(n_s, R0, t0, result, trace, corr);
    return PSULVSB_OK;
  }
  const psulvsb_icp_pair_t p = psulvsb::one_pair(src, n_s, tgt, n_t, tgt_normals, R0, t0);
  const psulvsb::Objective obj{psulvsb::GICP, &src_normals, 1.0 - epsilon};
  return psulvsb::run_icp_host(&p, 1, *params, obj, result, trace, corr, "psulvsb_gicp_host");
}

unsigned long long psulvsb_gicp_batch_workspace_bytes(const psulvsb_gicp_pair_t* pairs, int B) {
  if (B <= 0 || !pairs) return 0ull;
  std::vector<psulvsb_icp_pair_t> sizes((size_t)B);
  for (int b = 0; b < B; ++b) {
    if (pairs[b].n_s < 0 || pairs[b].n_t < 0) return 0ull;
    sizes[b].n_s = pairs[b].n_s;
    sizes[b].n_t = pairs[b].n_t;
  }
  return (unsigned long long)psulvsb::icp_layout(psulvsb::icp_sizes(sizes.data(), B), nullptr, nullptr);
}

int psulvsb_gicp_batch(void* stream, const psulvsb_gicp_pair_t* pairs, int B, const psulvsb_icp_params_t* params,
                       double epsilon, void* d_work, psulvsb_icp_result_t* d_results, psulvsb_icp_iteration_t* d_trace,
                       int* d_corr) {
  if (B < 0 || !psulvsb::gicp_params_ok(params, epsilon) || (B > 0 && (!pairs || !d_work || !d_results)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_gicp_batch: bad argument");
  std::vector<psulvsb_icp_pair_t> icp;
  std::vector<const double*> snrm;
  if (int rc = psulvsb::gicp_pairs(pairs, B, params, icp, snrm, "psulvsb_gicp_batch")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  const psulvsb::Objective obj{psulvsb::GICP, snrm.data(), 1.0 - epsilon};
  return psulvsb::run_icp((cudaStream_t)stream, icp.data(), B, *params, obj, d_work, d_results, d_trace, d_corr);
}

int psulvsb_gicp_batch_host(const psulvsb_gicp_pair_t* pairs, int B, const psulvsb_icp_params_t* params,
                            double epsilon, psulvsb_icp_result_t* results, psulvsb_icp_iteration_t* trace, int* corr) {
  if (B < 0 || !psulvsb::gicp_params_ok(params, epsilon) || (B > 0 && (!pairs || !results)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_gicp_batch_host: bad argument");
  std::vector<psulvsb_icp_pair_t> icp;
  std::vector<const double*> snrm;
  if (int rc = psulvsb::gicp_pairs(pairs, B, params, icp, snrm, "psulvsb_gicp_batch_host")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  const psulvsb::Objective obj{psulvsb::GICP, snrm.data(), 1.0 - epsilon};
  return psulvsb::run_icp_host(icp.data(), B, *params, obj, results, trace, corr, "psulvsb_gicp_batch_host");
}

}  // extern "C"
