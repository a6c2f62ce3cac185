// k8_features.cu -- correspondences from two raw clouds: radius normals, FPFH descriptors (33 bins), the two-way
// nearest neighbour in descriptor space and FGR's matcher (mutual / one-way lists, tuple test).  What upstream
// TEASER++ gets from teaser::FPFHEstimation (PCL NormalEstimation + FPFHEstimation) and teaser::Matcher (FLANN +
// FGR's AdvancedMatching) before it calls solve(src_cloud, tgt_cloud, correspondences).  DESIGN.md section 10 is
// the specification; oracle/features.py restates it in numpy.  Parity with PCL / FLANN is unpinned.
//
// Neighbourhoods come from a uniform grid of cell size h = max(r_n, r_f) (+1e-5 relative, so that a pair that
// passes the FP32 distance test is never two cells apart), hashed into nb = 2^ceil(log2 n) buckets: the workspace
// depends on n only.  Points of a bucket are stored contiguously in ascending index order (float4: x, y, z, index),
// so every walk -- the 27 cells around a point in a fixed order, a bucket visited once even when two cells share
// it -- sees its neighbours in one fixed order: every result is the same from call to call.  Hash collisions only
// add candidates; the distance test removes them.  No neighbour list is stored: each pass walks the cells again.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "eig3.cuh"
#include "ft_batch.cuh"
#include "grid.cuh"

namespace psulvsb {

namespace {

constexpr int FT_BINS = 11;
constexpr int FT_DIM = 33;

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

// ---- radius normals: FP64 mean and covariance of the r_n neighbourhood, smallest eigenvector, towards the viewpoint.
// kCap (hybrid): only the max_nn smallest keys of the neighbourhood count.  A first walk keeps them in shared memory
// ([slot][thread]: a warp's slot s is 32 consecutive words) and yields the threshold K* = the max_nn-th smallest key
// (all keys when the neighbourhood is no larger); the mean and covariance walks then skip keys above K*, so the sums
// run over the kept points in the radius mode's order.
template <bool kBatch, bool kCap = false>
__global__ void __launch_bounds__(FT_THREADS)
    k8_radius_normals(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one, const int* __restrict__ tile_first, int B, double inv_h,
                      const float4* __restrict__ spts, const int* __restrict__ start, float rn2,
                      double* __restrict__ normals, float4* __restrict__ nf, int max_nn = 0) {
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int p = first + threadIdx.x;
  if (p >= cl.n) return;
  const Grid g{inv_h, cl.mask, spts, start + cl.b0 + ci};
  const double* pts = cl.pts;
  const float4 me = spts[cl.p0 + p];
  const int i = __float_as_int(me.w);
  unsigned long long kstar = ~0ull;
  if constexpr (kCap) {
    __shared__ unsigned long long kept[FT_MAX_NN][FT_THREADS];
    const int tid = threadIdx.x;
    int nk = 0, top = 0;                 // candidates seen; the slot of the largest kept key
    unsigned long long kmax = 0;
    for_neighbours(g, me, rn2, [&](float4 q, int j) {
      const unsigned long long k = nn_key(me, q, j);
      if (nk < max_nn) {
        kept[nk][tid] = k;
        if (k > kmax) {
          kmax = k;
          top = nk;
        }
      } else if (k < kmax) {             // replace the largest, then find the new largest
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
    });
    if (nk > max_nn) kstar = kmax;
  }
  double mean[3] = {0, 0, 0};
  int cnt = 0;
  for_neighbours(g, me, rn2, [&](float4 q, int j) {
    if constexpr (kCap)
      if (nn_key(me, q, j) > kstar) return;
    for (int r = 0; r < 3; ++r) mean[r] += pts[3 * (size_t)j + r];
    ++cnt;
  });
  double nv[3];
  if (cnt < 3) {  // no plane through fewer than three points (PCL answers NaN)
    nv[0] = nv[1] = nv[2] = nan("");
  } else {
    for (int r = 0; r < 3; ++r) mean[r] /= (double)cnt;
    double cov[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for_neighbours(g, me, rn2, [&](float4 q, int j) {
      if constexpr (kCap)
        if (nn_key(me, q, j) > kstar) return;
      double d[3];
      for (int r = 0; r < 3; ++r) d[r] = pts[3 * (size_t)j + r] - mean[r];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) cov[r][c] += d[r] * d[c];
    });
    smallest_eigenvector(cov, nv);
    const double px = pts[3 * (size_t)i], py = pts[3 * (size_t)i + 1], pz = pts[3 * (size_t)i + 2];
    const double vx = cl.vp[0], vy = cl.vp[1], vz = cl.vp[2];
    if ((vx - px) * nv[0] + (vy - py) * nv[1] + (vz - pz) * nv[2] < 0.0) {  // flipNormalTowardsViewpoint
      nv[0] = -nv[0];
      nv[1] = -nv[1];
      nv[2] = -nv[2];
    }
  }
  const size_t o = (size_t)cl.p0 + i;
  if (normals)
    for (int r = 0; r < 3; ++r) normals[3 * o + r] = nv[r];
  nf[o] = make_float4((float)nv[0], (float)nv[1], (float)nv[2], 0.f);
}

__device__ __forceinline__ float dot3(float ax, float ay, float az, float bx, float by, float bz) {
  return __fadd_rn(__fadd_rn(__fmul_rn(ax, bx), __fmul_rn(ay, by)), __fmul_rn(az, bz));
}

__device__ __forceinline__ int feature_bin(double arg) {  // floor of the bin argument, clamped to [0, 10]
  const int b = (int)floor(arg);
  return b < 0 ? 0 : (b > FT_BINS - 1 ? FT_BINS - 1 : b);
}

// PCL computePairFeatures of (p, q) with d = q - p, in FP32; false = the pair is skipped
__device__ __forceinline__ bool pair_features(float4 p, float4 np, float4 q, float4 nq, float& f1, float& f2,
                                              float& f3) {
  if (isnan(np.x) || isnan(nq.x)) return false;
  float dx = q.x - p.x, dy = q.y - p.y, dz = q.z - p.z;
  const float len = __fsqrt_rn(dot3(dx, dy, dz, dx, dy, dz));
  if (len == 0.f) return false;
  const float a1 = __fdiv_rn(dot3(np.x, np.y, np.z, dx, dy, dz), len);
  const float a2 = __fdiv_rn(dot3(nq.x, nq.y, nq.z, dx, dy, dz), len);
  float4 n1 = np, n2 = nq;
  // acos(|a1|) > acos(|a2|) <=> |a1| < |a2| (acos decreases); the comparison does not depend on acos's rounding
  if (fabsf(a1) < fabsf(a2)) {
    n1 = nq;
    n2 = np;
    dx = -dx;
    dy = -dy;
    dz = -dz;
    f3 = -a2;
  } else {
    f3 = a1;
  }
  float vx = __fsub_rn(__fmul_rn(dy, n1.z), __fmul_rn(dz, n1.y));  // v = d x n1
  float vy = __fsub_rn(__fmul_rn(dz, n1.x), __fmul_rn(dx, n1.z));
  float vz = __fsub_rn(__fmul_rn(dx, n1.y), __fmul_rn(dy, n1.x));
  const float vn = __fsqrt_rn(dot3(vx, vy, vz, vx, vy, vz));
  if (vn == 0.f) return false;
  vx = __fdiv_rn(vx, vn);
  vy = __fdiv_rn(vy, vn);
  vz = __fdiv_rn(vz, vn);
  const float wx = __fsub_rn(__fmul_rn(n1.y, vz), __fmul_rn(n1.z, vy));  // w = n1 x v
  const float wy = __fsub_rn(__fmul_rn(n1.z, vx), __fmul_rn(n1.x, vz));
  const float wz = __fsub_rn(__fmul_rn(n1.x, vy), __fmul_rn(n1.y, vx));
  f2 = dot3(vx, vy, vz, n2.x, n2.y, n2.z);
  f1 = atan2f(dot3(wx, wy, wz, n2.x, n2.y, n2.z), dot3(n1.x, n1.y, n1.z, n2.x, n2.y, n2.z));
  return true;
}

// ---- SPFH: integer counts of the 3 x 11 bins over the pairs (i, j != i) of the r_f neighbourhood, and K_i
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS)
    k8_spfh(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one, const int* __restrict__ tile_first, int B, double inv_h,
            const float4* __restrict__ spts, const int* __restrict__ start, float rf2, const float4* __restrict__ nf,
            int* __restrict__ counts, int* __restrict__ kcount) {
  __shared__ int hist[FT_DIM][FT_THREADS];
  // a batch's grid and first point are read from shared memory at each use: held in registers across the walk they
  // push the kernel into spills
  __shared__ Grid s_grid;
  __shared__ volatile int s_p0;
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int p = first + threadIdx.x;
  const Grid one_grid{inv_h, cl.mask, spts, start};
  if constexpr (kBatch) {
    if (threadIdx.x == 0) {
      s_grid = Grid{inv_h, cl.mask, spts, start + cl.b0 + ci};
      s_p0 = cl.p0;
    }
    __syncthreads();
  }
  const Grid& g = kBatch ? s_grid : one_grid;
  auto p0 = [&]() { return kBatch ? (int)s_p0 : 0; };
  if (p >= cl.n) return;
  const int tid = threadIdx.x;
  for (int b = 0; b < FT_DIM; ++b) hist[b][tid] = 0;
  const float4 me = spts[p0() + p];
  const int i = __float_as_int(me.w);
  const float4 ni = nf[p0() + i];
  int K = 0;
  constexpr double kPi = 3.14159265358979323846;
  for_neighbours(g, me, rf2, [&](float4 q, int j) {
    ++K;
    float f1, f2, f3;
    if (j == i || !pair_features(me, ni, q, nf[p0() + j], f1, f2, f3)) return;
    hist[feature_bin(11.0 * ((double)f1 + kPi) / (2.0 * kPi))][tid] += 1;
    hist[FT_BINS + feature_bin(11.0 * ((double)f2 + 1.0) / 2.0)][tid] += 1;
    hist[2 * FT_BINS + feature_bin(11.0 * ((double)f3 + 1.0) / 2.0)][tid] += 1;
  });
  const size_t o = (size_t)p0() + i;
  for (int b = 0; b < FT_DIM; ++b) counts[o * FT_DIM + b] = hist[b][tid];
  kcount[o] = K;
}

// ---- FPFH: sum over neighbours j != i at distance > 0 of SPFH_j / |p_j - p_i|^2 (FP64), each 11 bins scaled to 100
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS)
    k8_fpfh(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one, const int* __restrict__ tile_first, int B, double inv_h,
            const float4* __restrict__ spts, const int* __restrict__ start, float rf2, const int* __restrict__ counts,
            const int* __restrict__ kcount, float* __restrict__ out) {
  __shared__ double acc[FT_DIM][FT_THREADS];
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int p = first + threadIdx.x;
  if (p >= cl.n) return;
  const Grid g{inv_h, cl.mask, spts, start + cl.b0 + ci};
  counts += (size_t)cl.p0 * FT_DIM;
  kcount += cl.p0;
  out += (size_t)cl.p0 * FT_DIM;
  const int tid = threadIdx.x;
  for (int b = 0; b < FT_DIM; ++b) acc[b][tid] = 0.0;
  const float4 me = spts[cl.p0 + p];
  const int i = __float_as_int(me.w);
  for_neighbours(g, me, rf2, [&](float4 q, int j) {
    const float d2 = sqdist(me, q);
    if (j == i || d2 == 0.f || kcount[j] < 2) return;
    const double w = (100.0 / (double)(kcount[j] - 1)) / (double)d2;
    for (int b = 0; b < FT_DIM; ++b) acc[b][tid] += (double)counts[(size_t)j * FT_DIM + b] * w;
  });
  for (int h = 0; h < 3; ++h) {
    double s = 0.0;
    for (int b = 0; b < FT_BINS; ++b) s += acc[h * FT_BINS + b][tid];
    for (int b = 0; b < FT_BINS; ++b)
      out[(size_t)i * FT_DIM + h * FT_BINS + b] = s > 0.0 ? (float)(acc[h * FT_BINS + b][tid] * (100.0 / s)) : 0.f;
  }
}

// ---- matcher batches: one pair on the device, the caller's psulvsb_match_pair_t and where it sits in the
// concatenations.  A pair with an empty side has ns = nt = 0: it takes no CTA, no list entry and no output.
struct FtPair {
  const double* src;
  const double* tgt;
  const float* fs;
  const float* ft;
  uint64_t seed;
  long long list0;  // first entry of its list (in the tuple test's workspace, else in the output)
  long long out0;   // first output pair: the caps of the pairs before it
  int ns, nt;
  int s0, t0;       // first source / target in the concatenations (row keys, nn_t, flags; column keys, nn_s)
  int rblocks;      // the NN's 256-row CTAs
};

// ---- two-way nearest neighbour over each pair's n_s x n_t matrix of squared L2 distances (difference form, FP32).
// A flat CTA index maps to (pair, 256-row block, 2048-column range) through the prefix of the pairs' CTA counts.
// A thread owns NN_ROWS source rows (in registers); a CTA walks one column range in tiles of 2 * NN_PAIRS target
// descriptors staged in shared memory as negated {column c, column c + 1} float2 pairs, so every dimension costs one
// FADD2 (the two differences) and one FFMA2 (the two squares into the two sums) per row.  Row minima stay in the
// thread (ascending columns, strict <: ties keep the lower column) and meet the other column ranges in a packed 64-bit
// atomicMin; column minima go warp -> CTA (shared memory) -> one packed atomicMin per column and CTA.  Key =
// (distance bits << 32) | index: non-negative float bits keep their order and the low word breaks ties.  Row keys and
// column keys are the concatenations over the pairs.
constexpr int NN_THREADS = 128;
constexpr int NN_ROWS = 2;
constexpr int NN_PAIRS = 32;
constexpr int NN_DP = 34;  // 33 dimensions padded to an even count (the pad is 0 on both sides)
constexpr int NN_COLS_PER_CTA = 2048;

template <bool kBatch>
__global__ void __launch_bounds__(NN_THREADS)
    k8_feature_nn(const FtPair* __restrict__ pairs, __grid_constant__ const FtPair one, const int* __restrict__ cta_first, int B,
                  unsigned long long* __restrict__ row_key, unsigned long long* __restrict__ col_key) {
  __shared__ __align__(16) float2 tile[NN_PAIRS][NN_DP];
  __shared__ unsigned long long wcol[NN_THREADS / 32][2 * NN_PAIRS];
  // a batch of one (kBatch false) takes its pair from the parameter `one` and a (row block, column range) grid
  int rblock = blockIdx.x, crange = blockIdx.y;
  FtPair pq = one;
  if constexpr (kBatch) {
    const int pi = pair_of(cta_first, B, blockIdx.x);
    pq = pairs[pi];
    const int cta = blockIdx.x - cta_first[pi];
    rblock = cta % pq.rblocks;
    crange = cta / pq.rblocks;
  }
  const float* __restrict__ fs = pq.fs;
  const float* __restrict__ ft = pq.ft;
  const int ns = pq.ns, nt = pq.nt;
  row_key += pq.s0;
  col_key += pq.t0;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int row0 = (rblock * NN_THREADS + tid) * NN_ROWS;  // lane-contiguous rows: lower lane = lower rows
  float a[NN_ROWS][NN_DP];
#pragma unroll
  for (int r = 0; r < NN_ROWS; ++r)
#pragma unroll
    for (int k = 0; k < NN_DP; ++k)
      a[r][k] = (row0 + r < ns && k < FT_DIM) ? fs[(size_t)(row0 + r) * FT_DIM + k] : 0.f;
  unsigned long long best[NN_ROWS];
#pragma unroll
  for (int r = 0; r < NN_ROWS; ++r) best[r] = ~0ull;
  const int c_begin = crange * NN_COLS_PER_CTA, c_end = min(nt, c_begin + NN_COLS_PER_CTA);
  for (int c0 = c_begin; c0 < c_end; c0 += 2 * NN_PAIRS) {
    __syncthreads();
    for (int e = tid; e < NN_PAIRS * NN_DP; e += NN_THREADS) {
      const int pr = e / NN_DP, k = e % NN_DP;
      const int ca = c0 + 2 * pr, cb = ca + 1;
      const float va = (ca < c_end && k < FT_DIM) ? ft[(size_t)ca * FT_DIM + k] : 0.f;
      const float vb = (cb < c_end && k < FT_DIM) ? ft[(size_t)cb * FT_DIM + k] : 0.f;
      tile[pr][k] = make_float2(-va, -vb);
    }
    __syncthreads();
    const int npairs = min(NN_PAIRS, (c_end - c0 + 1) / 2);
    for (int pr = 0; pr < npairs; ++pr) {
      float2 acc[NN_ROWS];
#pragma unroll
      for (int r = 0; r < NN_ROWS; ++r) acc[r] = make_float2(0.f, 0.f);
      const float4* t4 = reinterpret_cast<const float4*>(tile[pr]);
#pragma unroll
      for (int k2 = 0; k2 < NN_DP / 2; ++k2) {
        const float4 b = t4[k2];
#pragma unroll
        for (int r = 0; r < NN_ROWS; ++r) {
          const float2 d0 = add2(bc2(a[r][2 * k2]), make_float2(b.x, b.y));
          acc[r] = fma2(d0, d0, acc[r]);
          const float2 d1 = add2(bc2(a[r][2 * k2 + 1]), make_float2(b.z, b.w));
          acc[r] = fma2(d1, d1, acc[r]);
        }
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int c = c0 + 2 * pr + half;
        const bool cvalid = c < c_end;
        unsigned int cbest = 0xFFFFFFFFu;
        int crow = 0;
#pragma unroll
        for (int r = 0; r < NN_ROWS; ++r) {
          const float d = half ? acc[r].y : acc[r].x;
          const unsigned int bits = __float_as_uint(d);
          if (row0 + r < ns) {
            if (cvalid) {
              const unsigned long long key = ((unsigned long long)bits << 32) | (unsigned int)c;
              if (key < best[r]) best[r] = key;
            }
            if (bits < cbest) {
              cbest = bits;
              crow = row0 + r;
            }
          }
        }
        const unsigned int wbest = __reduce_min_sync(0xffffffffu, cbest);
        const unsigned int hit = __ballot_sync(0xffffffffu, cbest == wbest);
        const int wrow = __shfl_sync(0xffffffffu, crow, __ffs(hit) - 1);
        if (lane == 0)
          wcol[wid][2 * pr + half] =
              (cvalid && wbest != 0xFFFFFFFFu) ? (((unsigned long long)wbest << 32) | (unsigned int)wrow) : ~0ull;
      }
    }
    __syncthreads();
    for (int cc = tid; cc < 2 * npairs; cc += NN_THREADS) {
      unsigned long long k = wcol[0][cc];
      for (int w = 1; w < NN_THREADS / 32; ++w) k = min(k, wcol[w][cc]);
      if (k != ~0ull) atomicMin(col_key + c0 + cc, k);
    }
  }
#pragma unroll
  for (int r = 0; r < NN_ROWS; ++r)
    if (row0 + r < ns && best[r] != ~0ull) atomicMin(row_key + row0 + r, best[r]);
}

__global__ void k8_nn_finish(const unsigned long long* __restrict__ key, int n, int* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = key[i] == ~0ull ? -1 : (int)(unsigned int)key[i];
}

// ---- matcher list (FGR AdvancedMatching) over the concatenations: flag[i] for the first part, then one scan per pair
// places the pairs.  crosscheck: flag[i] = nn_s(nn_t(i)) == i.  one-way: flag[i] = i is nn_s(j) for some j (mark pass).
// nn_t[x] / nn_s[y] hold indices local to the pair.
__global__ void k8_match_flags(const FtPair* __restrict__ pairs, const int* __restrict__ s_first, int B, int NS,
                               const int* __restrict__ nn_t, const int* __restrict__ nn_s, int crosscheck,
                               const int* __restrict__ marked, int* __restrict__ flag) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= NS) return;
  const FtPair& pr = pairs[pair_of(s_first, B, x)];
  const int j = nn_t[x];
  flag[x] = crosscheck ? (j >= 0 && nn_s[pr.t0 + j] == x - pr.s0) : (marked[x] != 0 && j >= 0);
}

__global__ void k8_match_mark(const FtPair* __restrict__ pairs, const int* __restrict__ t_first, int B, int NT,
                              const int* __restrict__ nn_s, int* __restrict__ marked) {
  const int y = blockIdx.x * blockDim.x + threadIdx.x;
  if (y < NT && nn_s[y] >= 0) marked[pairs[pair_of(t_first, B, y)].s0 + nn_s[y]] = 1;
}

// one CTA per pair: pos[s0 + pair, s0 + pair + ns] = exclusive scan of the pair's flags; ncorr = the list's length.
// counts (may be NULL) receives ncorr, or 0 ahead of the tuple test.
__global__ void __launch_bounds__(SCAN_THREADS)
    k8_match_scan(const FtPair* __restrict__ pairs, const int* __restrict__ flag, int crosscheck, int tuple_test,
                  int* __restrict__ pos, int* __restrict__ ncorr, long long* __restrict__ counts) {
  const FtPair& pr = pairs[blockIdx.x];
  int* p = pos + pr.s0 + blockIdx.x;
  cta_scan(flag + pr.s0, pr.ns, p, nullptr, 0);
  if (threadIdx.x == 0) {
    const int n = p[pr.ns] + (crosscheck ? 0 : pr.nt);
    ncorr[blockIdx.x] = n;
    counts[blockIdx.x] = tuple_test ? 0 : n;
  }
}

// list[2k] = source index, list[2k + 1] = target index from the pair's list0; one thread per source of every pair,
// then (one-way lists) one per target: (nn_s(j), j) for every j after the flagged part
__global__ void k8_match_place(const FtPair* __restrict__ pairs, const int* __restrict__ s_first,
                               const int* __restrict__ t_first, int B, int NS, int NT, const int* __restrict__ nn_t,
                               const int* __restrict__ nn_s, int crosscheck, const int* __restrict__ flag,
                               const int* __restrict__ pos, int* __restrict__ list) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x < NS) {
    if (!flag[x]) return;
    const int p = pair_of(s_first, B, x);
    const FtPair& pr = pairs[p];
    const size_t k = (size_t)pr.list0 + pos[x + p];
    list[2 * k] = x - pr.s0;
    list[2 * k + 1] = nn_t[x];
  } else if (!crosscheck && x < NS + NT) {
    const int y = x - NS, p = pair_of(t_first, B, y);
    const FtPair& pr = pairs[p];
    const size_t k = (size_t)pr.list0 + pos[pr.s0 + p + pr.ns] + (y - pr.t0);
    list[2 * k] = nn_s[y];
    list[2 * k + 1] = y - pr.t0;
  }
}

// ---- tuple test: trial t draws list positions rand31(seed; TUPLE, 0, 3t + k) % ncorr, k = 0, 1, 2, and passes iff
// every source / target edge length ratio of the triangle lies strictly inside (s, 1/s) (FP32, FGR's expression).
// The kept set is the first 1000 passing trials among the first 100 ncorr, so the rounds' chunking cannot change it.
// Round r evaluates trials [r span, (r + 1) span) of every pair that is not done.
constexpr int TUPLE_THREADS = 256;

struct TupleState {
  int kept;
  int done;
};

__device__ __forceinline__ float len3(const double* __restrict__ P, int a, int b) {
  const float dx = (float)P[3 * (size_t)a] - (float)P[3 * (size_t)b];
  const float dy = (float)P[3 * (size_t)a + 1] - (float)P[3 * (size_t)b + 1];
  const float dz = (float)P[3 * (size_t)a + 2] - (float)P[3 * (size_t)b + 2];
  return __fsqrt_rn(dot3(dx, dy, dz, dx, dy, dz));
}

// one thread per (pair, trial of the round), `bpp` CTAs per pair: pass[pair * span + u]
__global__ void __launch_bounds__(TUPLE_THREADS)
    k8_tuple_trials(const FtPair* __restrict__ pairs, int bpp, int span, unsigned long long t0,
                    const TupleState* __restrict__ state, const int* __restrict__ ncorr, const int* __restrict__ lists,
                    float s, unsigned char* __restrict__ pass) {
  const int p = blockIdx.x / bpp, u = (blockIdx.x % bpp) * TUPLE_THREADS + threadIdx.x;
  if (u >= span) return;
  const size_t x = (size_t)p * span + u;
  const int n = ncorr[p];
  const unsigned long long t = t0 + u;
  if (state[p].done || t >= 100ull * (unsigned long long)n) return;
  const uint64_t seed = pairs[p].seed;
  const double *src = pairs[p].src, *tgt = pairs[p].tgt;
  const int* list = lists + 2 * pairs[p].list0;
  int r[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) r[k] = (int)(philox_rand31(seed, PSULVSB_DOMAIN_TUPLE, 0u, 3 * t + k) % (uint32_t)n);
  bool ok = true;
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    const int a = r[e], b = r[e == 2 ? 0 : e + 1];
    const float li = len3(src, list[2 * a], list[2 * b]);
    const float lj = len3(tgt, list[2 * a + 1], list[2 * b + 1]);
    ok = ok && (__fmul_rn(li, s) < lj) && (lj < __fdiv_rn(li, s));
  }
  pass[x] = ok ? 1 : 0;
}

// one CTA per pair: appends the passing trials of the round, in trial order, while fewer than max_tuples have been
// kept; a pair is done once it holds max_tuples or has run its 100 ncorr trials: counts[pair] = 3 kept, ndone += 1
__global__ void __launch_bounds__(SCAN_THREADS)
    k8_tuple_keep(const FtPair* __restrict__ pairs, int span, unsigned long long t0,
                  const unsigned char* __restrict__ pass, const int* __restrict__ ncorr, const int* __restrict__ lists,
                  int max_tuples, TupleState* __restrict__ state, int* __restrict__ ndone, int* __restrict__ outs,
                  long long* __restrict__ counts) {
  __shared__ int warp_tot[SCAN_THREADS / 32];
  __shared__ int base;
  const int p = blockIdx.x;
  TupleState* st = state + p;
  if (st->done) return;
  const FtPair& pr = pairs[p];
  const int n = ncorr[p];
  const unsigned long long trials = 100ull * (unsigned long long)n;
  const int nt = t0 >= trials ? 0 : (int)(trials - t0 < (unsigned long long)span ? trials - t0 : span);
  const int* list = lists + 2 * pr.list0;
  int* out = outs + 2 * pr.out0;
  pass += (size_t)p * span;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) base = st->kept;
  __syncthreads();
  for (int u0 = 0; u0 < nt && base < max_tuples; u0 += SCAN_THREADS) {
    const int u = u0 + tid;
    const int f = u < nt ? pass[u] : 0;
    const unsigned int bal = __ballot_sync(0xffffffffu, f);
    if (lane == 0) warp_tot[wid] = __popc(bal);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < SCAN_THREADS / 32; ++w) {
      before += w < wid ? warp_tot[w] : 0;
      total += warp_tot[w];
    }
    const int slot = base + before + __popc(bal & ((1u << lane) - 1u));
    if (f && slot < max_tuples) {
      const unsigned long long t = t0 + u;
      for (int k = 0; k < 3; ++k) {
        const int r = (int)(philox_rand31(pr.seed, PSULVSB_DOMAIN_TUPLE, 0u, 3 * t + k) % (uint32_t)n);
        out[2 * (3 * (size_t)slot + k)] = list[2 * r];
        out[2 * (3 * (size_t)slot + k) + 1] = list[2 * r + 1];
      }
    }
    __syncthreads();
    if (tid == 0) base = min(max_tuples, base + total);
    __syncthreads();
  }
  if (tid != 0) return;
  st->kept = base;
  if (base >= max_tuples || t0 + nt >= trials) {
    st->done = 1;
    counts[p] = 3ll * base;
    atomicAdd(ndone, 1);
  }
}

bool radius_ok(double r) { return std::isfinite(r) && r > 0.0; }

struct FpfhWork {
  FtCloud* cloud;   // [B], followed by tile_first [B + 1]: one copy uploads both
  int* tile_first;
  size_t table_bytes;
  float4 *spts, *nf;  // [n]: spts sorted by bucket, ascending index inside a bucket; .w = index in the cloud
  int *pbucket, *tmp, *kcount;  // [n]
  int *count, *cursor;          // [nb]
  int* start;                   // [nb + B]
  int* counts;                  // [33 n]
};

// the FPFH workspace; without descriptors (the normals stage alone) counts and kcount take no room
size_t fpfh_layout(const FpfhSizes& z, char* base, FpfhWork* w, bool descriptors = true) {
  const size_t nn = (size_t)z.n, nb = (size_t)z.nb, B = (size_t)z.B;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += up256(bytes);
    return p;
  };
  FpfhWork v;
  v.table_bytes = sizeof(FtCloud) * B + 4 * (B + 1);
  v.cloud = (FtCloud*)take(v.table_bytes);
  v.tile_first = (int*)((char*)v.cloud + sizeof(FtCloud) * B);
  v.spts = (float4*)take(16 * nn);
  v.nf = (float4*)take(16 * nn);
  v.pbucket = (int*)take(4 * nn);
  v.count = (int*)take(4 * nb);
  v.start = (int*)take(4 * (nb + B));
  v.cursor = (int*)take(4 * nb);
  v.tmp = (int*)take(4 * nn);
  v.counts = (int*)take(descriptors ? 4 * FT_DIM * nn : 0);
  v.kcount = (int*)take(descriptors ? 4 * nn : 0);
  if (w) *w = v;
  return off;
}

// features NULL: the normals stage alone, the first five launches (max_nn > 0: the hybrid neighbourhood)
template <bool kBatch>
void launch_fpfh(cudaStream_t st, const FpfhWork& w, const FtCloud& one, int B, int tiles, int n, double inv_h, float rn2,
                 float rf2, int max_nn, double* normals, float* features) {
  k8_grid_count<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, inv_h, w.pbucket, w.count);
  k8_cloud_scan<kBatch><<<B, SCAN_THREADS, 0, st>>>(w.cloud, one, w.count, w.start, w.cursor);
  k8_grid_scatter<<<blocks(n, GRID_THREADS), GRID_THREADS, 0, st>>>(n, w.pbucket, w.cursor, w.tmp);
  k8_grid_order<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, w.pbucket, w.start, w.tmp, w.spts);
  if (max_nn > 0) {
    k8_radius_normals<kBatch, true><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, inv_h, w.spts,
                                                                  w.start, rn2, normals, w.nf, max_nn);
    return;
  }
  k8_radius_normals<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, inv_h, w.spts, w.start, rn2,
                                                          normals, w.nf);
  if (!features) return;
  k8_spfh<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, inv_h, w.spts, w.start, rf2, w.nf,
                                                w.counts, w.kcount);
  k8_fpfh<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, inv_h, w.spts, w.start, rf2, w.counts,
                                                w.kcount, features);
}

// the batch on the device (clouds checked, B >= 1): one upload of the cloud table, then seven launches over all clouds.
// features NULL: the normals stage alone on the grid of cell size r_n (FPFH's grid whenever r_f <= r_n), five
// launches; max_nn: 0 for the radius neighbourhood, else the hybrid cap (normals only)
int run_fpfh(cudaStream_t st, const psulvsb_fpfh_cloud_t* clouds, int B, double rn, double rf, int max_nn, void* work,
             double* normals, float* features) {
  const FpfhSizes z = fpfh_sizes(clouds, B);
  if (z.tiles == 0) return PSULVSB_OK;
  FpfhWork w;
  fpfh_layout(z, static_cast<char*>(work), &w, features != nullptr);
  std::vector<char> table(w.table_bytes);
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
  if (B > 1) PSU_CUDA(cudaMemcpyAsync(w.cloud, table.data(), table.size(), cudaMemcpyHostToDevice, st));
  const double h = (rn > rf ? rn : rf) * (1.0 + 1e-5), inv_h = 1.0 / h;
  const int tiles = (int)z.tiles, n = (int)z.n;
  const float rn2 = (float)(rn * rn), rf2 = (float)(rf * rf);
  PSU_CUDA(cudaMemsetAsync(w.count, 0, 4 * (size_t)z.nb, st));
  if (B == 1)
    launch_fpfh<false>(st, w, hc[0], 1, tiles, n, inv_h, rn2, rf2, max_nn, normals, features);
  else
    launch_fpfh<true>(st, w, hc[0], B, tiles, n, inv_h, rn2, rf2, max_nn, normals, features);
  PSU_CHECK_LAUNCH(features ? "k8_fpfh" : "k8_radius_normals");
  return PSULVSB_OK;
}

// the batch on host buffers (clouds checked, B >= 1): the clouds go up in one copy, features and normals come back.
// features NULL: the normals stage alone (as run_fpfh)
int run_fpfh_host(const psulvsb_fpfh_cloud_t* clouds, int B, double rn, double rf, int max_nn, double* normals,
                  float* features, const char* who) {
  const FpfhSizes z = fpfh_sizes(clouds, B);
  if (z.n == 0) return PSULVSB_OK;
  const size_t N = (size_t)z.n, o_n = up256(features ? 4 * FT_DIM * N : 0),
               o_in = o_n + up256(normals ? 24 * N : 0), o_w = o_in + up256(24 * N);
  std::vector<char> in(B > 1 ? 24 * N : 0);
  std::vector<psulvsb_fpfh_cloud_t> dev(clouds, clouds + B);
  DevBuf buf;
  if (int rc = buf.alloc(o_w + fpfh_layout(z, nullptr, nullptr, features != nullptr), who)) return rc;
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
  if (int rc = run_fpfh(nullptr, dev.data(), B, rn, rf, max_nn, b + o_w, normals ? (double*)(b + o_n) : nullptr,
                        features ? (float*)b : nullptr))
    return rc;
  if (features) PSU_CUDA(cudaMemcpyAsync(features, b, 4 * FT_DIM * N, cudaMemcpyDeviceToHost, nullptr));
  if (normals) PSU_CUDA(cudaMemcpyAsync(normals, b + o_n, 24 * N, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaStreamSynchronize(nullptr));
  return PSULVSB_OK;
}

// ---- matcher batch on the host side
constexpr int MAX_TUPLES = 1000;
// trials of one tuple round over the whole batch, and the bounds of a pair's share: a single pair evaluates 2^20
// trials per round, a batch of 592 pairs 2^16 each
constexpr long long TUPLE_ROUND = 1ll << 26;
constexpr int TUPLE_CHUNK_MIN = 1 << 16, TUPLE_CHUNK_MAX = 1 << 20;

bool live(const psulvsb_match_pair_t& p) { return p.n_src > 0 && p.n_tgt > 0; }

long long list_cap(const psulvsb_match_pair_t& p, int crosscheck) {
  return live(p) ? (crosscheck ? p.n_src : (long long)p.n_src + p.n_tgt) : 0;
}

long long out_cap(const psulvsb_match_pair_t& p, int crosscheck, int tuple_test) {
  return !live(p) ? 0 : (tuple_test ? 3ll * MAX_TUPLES : list_cap(p, crosscheck));
}

struct MatchSizes {
  long long ns = 0, nt = 0, ctas = 0, list = 0, out = 0, max_list = 0;
  int B = 0, span = 0;  // span: trials per pair and tuple round (0 without the tuple test)
};

MatchSizes match_sizes(const psulvsb_match_pair_t* pairs, int B, int crosscheck, int tuple_test) {
  MatchSizes z;
  z.B = B;
  for (int b = 0; b < B; ++b) {
    const psulvsb_match_pair_t& p = pairs[b];
    z.out += out_cap(p, crosscheck, tuple_test);
    if (!live(p)) continue;
    z.ns += p.n_src;
    z.nt += p.n_tgt;
    z.ctas += (long long)blocks(p.n_src, NN_THREADS * NN_ROWS) * blocks(p.n_tgt, NN_COLS_PER_CTA);
    z.list += list_cap(p, crosscheck);
    z.max_list = std::max(z.max_list, list_cap(p, crosscheck));
  }
  if (tuple_test && z.max_list > 0) {
    long long chunk = TUPLE_CHUNK_MAX;
    while (chunk > TUPLE_CHUNK_MIN && chunk * B > TUPLE_ROUND) chunk >>= 1;
    z.span = (int)std::min(chunk, 100 * z.max_list);
  }
  return z;
}

struct MatchWork {
  FtPair* pair;  // [B], followed by cta_first, s_first, t_first [B + 1] each: one copy uploads the four
  int *cta_first, *s_first, *t_first;
  size_t table_bytes;
  unsigned long long* key;  // [ns + nt]: row keys, then column keys
  int* nn;                  // [ns + nt]: nn_t (source -> target), then nn_s
  int *mark, *flag;         // [ns]
  int* pos;                 // [ns + B]: pair p's scan at s0 + p, ns + 1 entries
  int* ncorr;               // [B]
  TupleState* state;        // [B], followed by ndone: one memset clears both
  int* ndone;
  int* list;                // [2 list] (tuple test)
  unsigned char* pass;      // [B span] (tuple test)
};

size_t match_layout(const MatchSizes& z, char* base, MatchWork* w) {
  const size_t B = (size_t)z.B, NS = (size_t)z.ns, NT = (size_t)z.nt;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += up256(bytes);
    return p;
  };
  MatchWork v;
  v.table_bytes = sizeof(FtPair) * B + 3 * 4 * (B + 1);
  v.pair = (FtPair*)take(v.table_bytes);
  v.cta_first = (int*)((char*)v.pair + sizeof(FtPair) * B);
  v.s_first = v.cta_first + (B + 1);
  v.t_first = v.s_first + (B + 1);
  v.key = (unsigned long long*)take(8 * (NS + NT));
  v.nn = (int*)take(4 * (NS + NT));
  v.mark = (int*)take(4 * NS);
  v.flag = (int*)take(4 * NS);
  v.pos = (int*)take(4 * (NS + B));
  v.ncorr = (int*)take(4 * B);
  v.state = (TupleState*)take(sizeof(TupleState) * B + 4);
  v.ndone = (int*)(v.state + B);
  v.list = (int*)take(z.span ? 8 * (size_t)z.list : 0);
  v.pass = (unsigned char*)take((size_t)z.span * B);
  if (w) *w = v;
  return off;
}

int match_check(const psulvsb_match_pair_t* pairs, int B, const char* who) {
  long long ns = 0, nt = 0;
  for (int b = 0; b < B; ++b) {
    const psulvsb_match_pair_t& p = pairs[b];
    if (p.n_src < 0 || p.n_tgt < 0 || (p.n_src > 0 && (!p.src || !p.fs)) || (p.n_tgt > 0 && (!p.tgt || !p.ft)))
      return fail(PSULVSB_ERR_INVALID, std::string(who) + ": bad pair " + std::to_string(b));
    ns += p.n_src;
    nt += p.n_tgt;
  }
  if (ns >= (1ll << 31) || nt >= (1ll << 31))
    return fail(PSULVSB_ERR_UNSUPPORTED, std::string(who) + ": the batch's clouds exceed 2^31 - 1 points in all");
  return PSULVSB_OK;
}

// the batch on the device (pairs checked, B >= 1): one upload of the pair table, the NN, the list and the tuple rounds.
// poll: wait for the stream after every tuple round and stop once every pair is done (the host variants); otherwise
// all ceil(100 max_list / span) rounds are issued without a host round trip.
int run_match(cudaStream_t st, const psulvsb_match_pair_t* pairs, int B, int crosscheck, int tuple_test,
              double tuple_scale, void* work, int* d_pairs, long long* d_counts, bool poll) {
  const MatchSizes z = match_sizes(pairs, B, crosscheck, tuple_test);
  MatchWork w;
  match_layout(z, static_cast<char*>(work), &w);
  std::vector<char> table(w.table_bytes);
  FtPair* hp = reinterpret_cast<FtPair*>(table.data());
  int* cta_first = reinterpret_cast<int*>(table.data() + sizeof(FtPair) * (size_t)B);
  int *s_first = cta_first + (B + 1), *t_first = s_first + (B + 1);
  cta_first[0] = s_first[0] = t_first[0] = 0;
  long long list0 = 0, out0 = 0;
  for (int b = 0; b < B; ++b) {
    const psulvsb_match_pair_t& q = pairs[b];
    FtPair& h = hp[b];
    h = FtPair{};
    const bool on = live(q);
    h.src = q.src;
    h.tgt = q.tgt;
    h.fs = q.fs;
    h.ft = q.ft;
    h.seed = q.seed;
    h.ns = on ? q.n_src : 0;
    h.nt = on ? q.n_tgt : 0;
    h.s0 = s_first[b];
    h.t0 = t_first[b];
    h.rblocks = on ? blocks(q.n_src, NN_THREADS * NN_ROWS) : 1;
    h.out0 = out0;
    h.list0 = tuple_test ? list0 : out0;
    out0 += out_cap(q, crosscheck, tuple_test);
    list0 += list_cap(q, crosscheck);
    cta_first[b + 1] = cta_first[b] + (on ? h.rblocks * blocks(q.n_tgt, NN_COLS_PER_CTA) : 0);
    s_first[b + 1] = s_first[b] + h.ns;
    t_first[b + 1] = t_first[b] + h.nt;
  }
  PSU_CUDA(cudaMemcpyAsync(w.pair, table.data(), table.size(), cudaMemcpyHostToDevice, st));
  const int NS = (int)z.ns, NT = (int)z.nt;
  int *nn_t = w.nn, *nn_s = w.nn + NS;
  if (z.ctas > 0) {
    PSU_CUDA(cudaMemsetAsync(w.key, 0xFF, 8 * ((size_t)NS + NT), st));
    if (B == 1)
      k8_feature_nn<false><<<dim3(hp[0].rblocks, blocks(NT, NN_COLS_PER_CTA)), NN_THREADS, 0, st>>>(
          w.pair, hp[0], w.cta_first, 1, w.key, w.key + NS);
    else
      k8_feature_nn<true><<<(int)z.ctas, NN_THREADS, 0, st>>>(w.pair, hp[0], w.cta_first, B, w.key, w.key + NS);
    PSU_CHECK_LAUNCH("k8_feature_nn");
    k8_nn_finish<<<blocks((long long)NS + NT, 256), 256, 0, st>>>(w.key, NS + NT, w.nn);
    PSU_CHECK_LAUNCH("k8_nn_finish");
    if (!crosscheck) {
      PSU_CUDA(cudaMemsetAsync(w.mark, 0, 4 * (size_t)NS, st));
      k8_match_mark<<<blocks(NT, 256), 256, 0, st>>>(w.pair, w.t_first, B, NT, nn_s, w.mark);
      PSU_CHECK_LAUNCH("k8_match_mark");
    }
    k8_match_flags<<<blocks(NS, 256), 256, 0, st>>>(w.pair, w.s_first, B, NS, nn_t, nn_s, crosscheck, w.mark, w.flag);
    PSU_CHECK_LAUNCH("k8_match_flags");
  }
  k8_match_scan<<<B, SCAN_THREADS, 0, st>>>(w.pair, w.flag, crosscheck, tuple_test, w.pos, w.ncorr, d_counts);
  PSU_CHECK_LAUNCH("k8_match_scan");
  if (z.ctas == 0) return PSULVSB_OK;
  int* list = tuple_test ? w.list : d_pairs;
  const long long nplace = (long long)NS + (crosscheck ? 0 : NT);
  k8_match_place<<<blocks(nplace, 256), 256, 0, st>>>(w.pair, w.s_first, w.t_first, B, NS, NT, nn_t, nn_s, crosscheck,
                                                      w.flag, w.pos, list);
  PSU_CHECK_LAUNCH("k8_match_place");
  if (!tuple_test) return PSULVSB_OK;
  PSU_CUDA(cudaMemsetAsync(w.state, 0, sizeof(TupleState) * (size_t)B + 4, st));
  const long long span = z.span, rounds = (100 * z.max_list + span - 1) / span;
  const int bpp = blocks(span, TUPLE_THREADS);
  for (long long r = 0; r < rounds; ++r) {
    const unsigned long long t0 = (unsigned long long)(r * span);
    k8_tuple_trials<<<bpp * B, TUPLE_THREADS, 0, st>>>(w.pair, bpp, (int)span, t0, w.state, w.ncorr, w.list,
                                                       (float)tuple_scale, w.pass);
    PSU_CHECK_LAUNCH("k8_tuple_trials");
    k8_tuple_keep<<<B, SCAN_THREADS, 0, st>>>(w.pair, (int)span, t0, w.pass, w.ncorr, w.list, MAX_TUPLES, w.state,
                                              w.ndone, d_pairs, d_counts);
    PSU_CHECK_LAUNCH("k8_tuple_keep");
    if (poll) {
      int done = 0;
      PSU_CUDA(cudaMemcpyAsync(&done, w.ndone, 4, cudaMemcpyDeviceToHost, st));
      PSU_CUDA(cudaStreamSynchronize(st));
      if (done == B) break;
    }
  }
  return PSULVSB_OK;
}

// the batch on host buffers (pairs checked, B >= 1): the live pairs' points and descriptors go up in one copy into
// `buf`, which then holds counts [B] (long long) and the pairs (Σ cap) from offset 0, ready to come back
int run_match_host(const psulvsb_match_pair_t* pairs, int B, int crosscheck, int tuple_test, double tuple_scale,
                   DevBuf& buf, const char* who) {
  const MatchSizes z = match_sizes(pairs, B, crosscheck, tuple_test);
  const size_t o_pairs = 8 * (size_t)B, o_in = up256(o_pairs + 8 * (size_t)z.out);
  // the live pairs' src, tgt, fs, ft in pair order, each pair's block 8-byte aligned
  std::vector<psulvsb_match_pair_t> dev(pairs, pairs + B);
  std::vector<size_t> in_off(B);
  size_t in_bytes = 0;
  for (int b = 0; b < B; ++b) {
    in_off[b] = in_bytes;
    if (live(dev[b])) in_bytes += ((24 + 4 * FT_DIM) * ((size_t)dev[b].n_src + dev[b].n_tgt) + 7) & ~size_t(7);
  }
  const size_t o_work = up256(o_in + in_bytes);
  if (int rc = buf.alloc(o_work + match_layout(z, nullptr, nullptr), who)) return rc;
  char* base = static_cast<char*>(buf.p);
  // a single pair's four arrays go up straight from the caller's buffers: packing them first would only add a host copy
  std::vector<char> in(B > 1 ? in_bytes : 0);
  for (int b = 0; b < B; ++b) {
    psulvsb_match_pair_t& q = dev[b];
    if (!live(q)) continue;
    size_t off = in_off[b];
    auto put = [&](const void* h, size_t bytes) -> const char* {
      char* d = base + o_in + off;
      if (B > 1)
        std::memcpy(in.data() + off, h, bytes);
      else if (cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, nullptr) != cudaSuccess)
        return nullptr;
      off += bytes;
      return d;
    };
    const size_t ns = (size_t)q.n_src, nt = (size_t)q.n_tgt;
    q.src = (const double*)put(q.src, 24 * ns);
    q.tgt = (const double*)put(q.tgt, 24 * nt);
    q.fs = (const float*)put(q.fs, 4 * FT_DIM * ns);
    q.ft = (const float*)put(q.ft, 4 * FT_DIM * nt);
    if (!q.src || !q.tgt || !q.fs || !q.ft) return fail(PSULVSB_ERR_CUDA, std::string(who) + ": copy in failed");
  }
  if (B > 1 && in_bytes) PSU_CUDA(cudaMemcpyAsync(base + o_in, in.data(), in_bytes, cudaMemcpyHostToDevice, nullptr));
  return run_match(nullptr, dev.data(), B, crosscheck, tuple_test, tuple_scale, base + o_work, (int*)(base + o_pairs),
                   (long long*)base, true);
}

}  // namespace

}  // namespace psulvsb

using psulvsb::fail;

extern "C" {

unsigned long long psulvsb_fpfh_workspace_bytes(int n) {
  if (n < 0) return 0ull;
  const psulvsb_fpfh_cloud_t c{nullptr, n, {0.0, 0.0, 0.0}};
  return (unsigned long long)psulvsb::fpfh_layout(psulvsb::fpfh_sizes(&c, 1), nullptr, nullptr);
}

unsigned long long psulvsb_fpfh_batch_workspace_bytes(const psulvsb_fpfh_cloud_t* clouds, int B) {
  if (B <= 0 || !clouds) return 0ull;
  for (int c = 0; c < B; ++c)
    if (clouds[c].n < 0) return 0ull;
  return (unsigned long long)psulvsb::fpfh_layout(psulvsb::fpfh_sizes(clouds, B), nullptr, nullptr);
}

static psulvsb_fpfh_cloud_t one_cloud(const double* pts, int n, const double viewpoint[3]) {
  psulvsb_fpfh_cloud_t c{pts, n, {0.0, 0.0, 0.0}};
  if (viewpoint)
    for (int r = 0; r < 3; ++r) c.viewpoint[r] = viewpoint[r];
  return c;
}

int psulvsb_fpfh(void* stream, const double* d_pts, int n, double normal_radius, double feature_radius,
                 const double viewpoint[3], void* d_work, double* d_normals, float* d_features) {
  if (n < 0 || !psulvsb::radius_ok(normal_radius) || !psulvsb::radius_ok(feature_radius) ||
      (n > 0 && (!d_pts || !d_work || !d_features)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_fpfh: bad argument (radii must be finite and > 0)");
  if (int rc = psulvsb::need_device()) return rc;
  const psulvsb_fpfh_cloud_t c = one_cloud(d_pts, n, viewpoint);
  return psulvsb::run_fpfh((cudaStream_t)stream, &c, 1, normal_radius, feature_radius, 0, d_work, d_normals,
                           d_features);
}

int psulvsb_fpfh_host(const double* pts, int n, double normal_radius, double feature_radius, const double viewpoint[3],
                      double* normals, float* features) {
  if (n < 0 || !psulvsb::radius_ok(normal_radius) || !psulvsb::radius_ok(feature_radius) ||
      (n > 0 && (!pts || !features)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_fpfh_host: bad argument (radii must be finite and > 0)");
  if (int rc = psulvsb::need_device()) return rc;
  const psulvsb_fpfh_cloud_t c = one_cloud(pts, n, viewpoint);
  return psulvsb::run_fpfh_host(&c, 1, normal_radius, feature_radius, 0, normals, features, "psulvsb_fpfh_host");
}

int psulvsb_fpfh_batch(void* stream, const psulvsb_fpfh_cloud_t* clouds, int B, double normal_radius,
                       double feature_radius, void* d_work, double* d_normals, float* d_features) {
  if (B < 0 || !psulvsb::radius_ok(normal_radius) || !psulvsb::radius_ok(feature_radius) ||
      (B > 0 && (!clouds || !d_work || !d_features)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_fpfh_batch: bad argument (radii must be finite and > 0)");
  if (int rc = psulvsb::clouds_check(clouds, B, "psulvsb_fpfh_batch")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_fpfh((cudaStream_t)stream, clouds, B, normal_radius, feature_radius, 0, d_work, d_normals,
                           d_features);
}

int psulvsb_fpfh_batch_host(const psulvsb_fpfh_cloud_t* clouds, int B, double normal_radius, double feature_radius,
                            double* normals, float* features) {
  if (B < 0 || !psulvsb::radius_ok(normal_radius) || !psulvsb::radius_ok(feature_radius) ||
      (B > 0 && (!clouds || !features)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_fpfh_batch_host: bad argument (radii must be finite and > 0)");
  if (int rc = psulvsb::clouds_check(clouds, B, "psulvsb_fpfh_batch_host")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_fpfh_host(clouds, B, normal_radius, feature_radius, 0, normals, features,
                                "psulvsb_fpfh_batch_host");
}

// ---- normals alone (DESIGN.md section 10, "Normals alone"): FPFH's grid and normals kernel, nothing after them
static bool max_nn_ok(int max_nn) { return max_nn == 0 || (max_nn >= 3 && max_nn <= psulvsb::FT_MAX_NN); }

unsigned long long psulvsb_normals_workspace_bytes(int n) {
  if (n < 0) return 0ull;
  const psulvsb_fpfh_cloud_t c{nullptr, n, {0.0, 0.0, 0.0}};
  return (unsigned long long)psulvsb::fpfh_layout(psulvsb::fpfh_sizes(&c, 1), nullptr, nullptr, false);
}

unsigned long long psulvsb_normals_batch_workspace_bytes(const psulvsb_fpfh_cloud_t* clouds, int B) {
  if (B <= 0 || !clouds) return 0ull;
  for (int c = 0; c < B; ++c)
    if (clouds[c].n < 0) return 0ull;
  return (unsigned long long)psulvsb::fpfh_layout(psulvsb::fpfh_sizes(clouds, B), nullptr, nullptr, false);
}

int psulvsb_normals(void* stream, const double* d_pts, int n, double radius, int max_nn, const double viewpoint[3],
                    void* d_work, double* d_normals) {
  if (n < 0 || !psulvsb::radius_ok(radius) || !max_nn_ok(max_nn) || (n > 0 && (!d_pts || !d_work || !d_normals)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_normals: bad argument (radius finite and > 0, max_nn 0 or 3..32)");
  const psulvsb_fpfh_cloud_t c = one_cloud(d_pts, n, viewpoint);
  if (int rc = psulvsb::clouds_check(&c, 1, "psulvsb_normals")) return rc;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_fpfh((cudaStream_t)stream, &c, 1, radius, radius, max_nn, d_work, d_normals, nullptr);
}

int psulvsb_normals_host(const double* pts, int n, double radius, int max_nn, const double viewpoint[3],
                         double* normals) {
  if (n < 0 || !psulvsb::radius_ok(radius) || !max_nn_ok(max_nn) || (n > 0 && (!pts || !normals)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_normals_host: bad argument (radius finite and > 0, max_nn 0 or 3..32)");
  const psulvsb_fpfh_cloud_t c = one_cloud(pts, n, viewpoint);
  if (int rc = psulvsb::clouds_check(&c, 1, "psulvsb_normals_host")) return rc;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_fpfh_host(&c, 1, radius, radius, max_nn, normals, nullptr, "psulvsb_normals_host");
}

int psulvsb_normals_batch(void* stream, const psulvsb_fpfh_cloud_t* clouds, int B, double radius, int max_nn,
                          void* d_work, double* d_normals) {
  if (B < 0 || !psulvsb::radius_ok(radius) || !max_nn_ok(max_nn) || (B > 0 && (!clouds || !d_work || !d_normals)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_normals_batch: bad argument (radius finite and > 0, max_nn 0 or 3..32)");
  if (int rc = psulvsb::clouds_check(clouds, B, "psulvsb_normals_batch")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_fpfh((cudaStream_t)stream, clouds, B, radius, radius, max_nn, d_work, d_normals, nullptr);
}

int psulvsb_normals_batch_host(const psulvsb_fpfh_cloud_t* clouds, int B, double radius, int max_nn,
                               double* normals) {
  if (B < 0 || !psulvsb::radius_ok(radius) || !max_nn_ok(max_nn) || (B > 0 && (!clouds || !normals)))
    return fail(PSULVSB_ERR_INVALID,
                "psulvsb_normals_batch_host: bad argument (radius finite and > 0, max_nn 0 or 3..32)");
  if (int rc = psulvsb::clouds_check(clouds, B, "psulvsb_normals_batch_host")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_fpfh_host(clouds, B, radius, radius, max_nn, normals, nullptr, "psulvsb_normals_batch_host");
}

int psulvsb_feature_nn(void* stream, const float* d_fs, int n_src, const float* d_ft, int n_tgt, int* d_nn_src_to_tgt,
                       int* d_nn_tgt_to_src) {
  if (n_src < 0 || n_tgt < 0 || (n_src > 0 && (!d_fs || !d_nn_src_to_tgt)) || (n_tgt > 0 && (!d_ft || !d_nn_tgt_to_src)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_feature_nn: bad argument");
  if (int rc = psulvsb::need_device()) return rc;
  using namespace psulvsb;
  cudaStream_t st = (cudaStream_t)stream;
  if (n_src == 0 && n_tgt == 0) return PSULVSB_OK;
  if (n_src == 0 || n_tgt == 0) {  // nothing to be near to
    if (n_src) PSU_CUDA(cudaMemsetAsync(d_nn_src_to_tgt, 0xFF, 4 * (size_t)n_src, st));
    if (n_tgt) PSU_CUDA(cudaMemsetAsync(d_nn_tgt_to_src, 0xFF, 4 * (size_t)n_tgt, st));
    return PSULVSB_OK;
  }
  // a batch of one: the pair travels as a kernel parameter, the keys in the call's own allocation
  FtPair one{};
  one.fs = d_fs;
  one.ft = d_ft;
  one.ns = n_src;
  one.nt = n_tgt;
  one.rblocks = blocks(n_src, NN_THREADS * NN_ROWS);
  const size_t nk = (size_t)n_src + (size_t)n_tgt;
  unsigned long long* keys = nullptr;
  PSU_CUDA(cudaMallocAsync((void**)&keys, 8 * nk, st));
  int rc = PSULVSB_OK;
  if (cudaMemsetAsync(keys, 0xFF, 8 * nk, st) != cudaSuccess) rc = fail(PSULVSB_ERR_CUDA, "feature nn: memset failed");
  if (!rc) {
    k8_feature_nn<false><<<dim3(one.rblocks, blocks(n_tgt, NN_COLS_PER_CTA)), NN_THREADS, 0, st>>>(nullptr, one, nullptr,
                                                                                                  1, keys, keys + n_src);
    if (cudaGetLastError() != cudaSuccess) rc = fail(PSULVSB_ERR_CUDA, "k8_feature_nn launch failed");
  }
  if (!rc) {
    k8_nn_finish<<<blocks(n_src, 256), 256, 0, st>>>(keys, n_src, d_nn_src_to_tgt);
    k8_nn_finish<<<blocks(n_tgt, 256), 256, 0, st>>>(keys + n_src, n_tgt, d_nn_tgt_to_src);
    if (cudaGetLastError() != cudaSuccess) rc = fail(PSULVSB_ERR_CUDA, "k8_nn_finish launch failed");
  }
  cudaFreeAsync(keys, st);
  return rc;
}

int psulvsb_match_host(const double* src_pts, int n_src, const double* tgt_pts, int n_tgt, const float* fs,
                       const float* ft, int crosscheck, int tuple_test, double tuple_scale, uint64_t seed, int* pairs,
                       long long capacity, long long* n_pairs) {
  if (!n_pairs || n_src < 0 || n_tgt < 0 || capacity < 0 || (capacity > 0 && !pairs) ||
      (n_src > 0 && (!src_pts || !fs)) || (n_tgt > 0 && (!tgt_pts || !ft)) || (tuple_test && !std::isfinite(tuple_scale)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_match_host: bad argument");
  *n_pairs = 0;
  if (int rc = psulvsb::need_device()) return rc;
  if (n_src == 0 || n_tgt == 0) return PSULVSB_OK;
  const psulvsb_match_pair_t p{src_pts, n_src, tgt_pts, n_tgt, fs, ft, seed};
  psulvsb::DevBuf buf;
  if (int rc = psulvsb::run_match_host(&p, 1, crosscheck, tuple_test, tuple_scale, buf, "psulvsb_match_host")) return rc;
  long long count = 0;
  PSU_CUDA(cudaMemcpyAsync(&count, buf.p, 8, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaStreamSynchronize(nullptr));
  *n_pairs = count;
  if (count > capacity)
    return fail(PSULVSB_ERR_CAPACITY, "psulvsb_match_host: " + std::to_string(count) + " pairs, capacity " +
                                          std::to_string(capacity));
  if (count) PSU_CUDA(cudaMemcpyAsync(pairs, (char*)buf.p + 8, 8 * (size_t)count, cudaMemcpyDeviceToHost, nullptr));
  PSU_CUDA(cudaStreamSynchronize(nullptr));
  return PSULVSB_OK;
}

unsigned long long psulvsb_match_batch_workspace_bytes(const psulvsb_match_pair_t* pairs, int B, int crosscheck,
                                                       int tuple_test) {
  if (B <= 0 || !pairs) return 0ull;
  for (int b = 0; b < B; ++b)
    if (pairs[b].n_src < 0 || pairs[b].n_tgt < 0) return 0ull;
  return (unsigned long long)psulvsb::match_layout(psulvsb::match_sizes(pairs, B, crosscheck, tuple_test), nullptr,
                                                   nullptr);
}

int psulvsb_match_batch(void* stream, const psulvsb_match_pair_t* pairs, int B, int crosscheck, int tuple_test,
                        double tuple_scale, void* d_work, int* d_pairs, long long* d_counts) {
  if (B < 0 || (tuple_test && !std::isfinite(tuple_scale)) || (B > 0 && (!pairs || !d_work || !d_pairs || !d_counts)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_match_batch: bad argument");
  if (int rc = psulvsb::match_check(pairs, B, "psulvsb_match_batch")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_match((cudaStream_t)stream, pairs, B, crosscheck, tuple_test, tuple_scale, d_work, d_pairs,
                            d_counts, false);
}

int psulvsb_match_batch_host(const psulvsb_match_pair_t* pairs, int B, int crosscheck, int tuple_test,
                             double tuple_scale, int* pairs_out, long long* counts) {
  if (B < 0 || (tuple_test && !std::isfinite(tuple_scale)) || (B > 0 && (!pairs || !pairs_out || !counts)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_match_batch_host: bad argument");
  if (int rc = psulvsb::match_check(pairs, B, "psulvsb_match_batch_host")) return rc;
  if (B == 0) return PSULVSB_OK;
  if (int rc = psulvsb::need_device()) return rc;
  psulvsb::DevBuf buf;
  if (int rc = psulvsb::run_match_host(pairs, B, crosscheck, tuple_test, tuple_scale, buf, "psulvsb_match_batch_host"))
    return rc;
  const psulvsb::MatchSizes z = psulvsb::match_sizes(pairs, B, crosscheck, tuple_test);
  PSU_CUDA(cudaMemcpyAsync(counts, buf.p, 8 * (size_t)B, cudaMemcpyDeviceToHost, nullptr));
  if (z.out) PSU_CUDA(cudaMemcpyAsync(pairs_out, (char*)buf.p + 8 * (size_t)B, 8 * (size_t)z.out, cudaMemcpyDeviceToHost,
                                      nullptr));
  PSU_CUDA(cudaStreamSynchronize(nullptr));
  return PSULVSB_OK;
}

}  // extern "C"
