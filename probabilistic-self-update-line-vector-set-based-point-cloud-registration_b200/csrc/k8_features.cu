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

#include <cmath>
#include <string>

#include "common.cuh"
#include "eig3.cuh"
#include "grid.cuh"

namespace psulvsb {

namespace {

constexpr int FT_THREADS = 128;
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

// ---- grid build: count, scan, scatter, order (each bucket's members ascending by index)
__global__ void __launch_bounds__(FT_THREADS)
    k8_grid_count(const double* __restrict__ pts, int n, double inv_h, unsigned int mask, int* __restrict__ pbucket,
                  int* __restrict__ count) {
  const int i = blockIdx.x * FT_THREADS + threadIdx.x;
  if (i >= n) return;
  const float x = (float)pts[3 * (size_t)i], y = (float)pts[3 * (size_t)i + 1], z = (float)pts[3 * (size_t)i + 2];
  const unsigned int b = bucket_of(cell_of(x, inv_h), cell_of(y, inv_h), cell_of(z, inv_h), mask);
  pbucket[i] = (int)b;
  atomicAdd(count + b, 1);
}

// the scatter's order inside a bucket depends on timing: rank each member by index instead
__global__ void __launch_bounds__(FT_THREADS)
    k8_grid_order(const double* __restrict__ pts, int n, const int* __restrict__ pbucket, const int* __restrict__ start,
                  const int* __restrict__ tmp, float4* __restrict__ spts) {
  const int p = blockIdx.x * FT_THREADS + threadIdx.x;
  if (p >= n) return;
  const int i = tmp[p];
  const int b = pbucket[i], s0 = start[b], s1 = start[b + 1];
  int rank = 0;
  for (int q = s0; q < s1; ++q) rank += tmp[q] < i;
  spts[s0 + rank] = make_float4((float)pts[3 * (size_t)i], (float)pts[3 * (size_t)i + 1],
                                (float)pts[3 * (size_t)i + 2], __int_as_float(i));
}

// ---- radius normals: FP64 mean and covariance of the r_n neighbourhood, smallest eigenvector, towards the viewpoint
__global__ void __launch_bounds__(FT_THREADS)
    k8_radius_normals(Grid g, const double* __restrict__ pts, int n, float rn2, double vx, double vy, double vz,
                      double* __restrict__ normals, float4* __restrict__ nf) {
  const int p = blockIdx.x * FT_THREADS + threadIdx.x;
  if (p >= n) return;
  const float4 me = g.spts[p];
  const int i = __float_as_int(me.w);
  double mean[3] = {0, 0, 0};
  int cnt = 0;
  for_neighbours(g, me, rn2, [&](float4, int j) {
    for (int r = 0; r < 3; ++r) mean[r] += pts[3 * (size_t)j + r];
    ++cnt;
  });
  double nv[3];
  if (cnt < 3) {  // no plane through fewer than three points (PCL answers NaN)
    nv[0] = nv[1] = nv[2] = nan("");
  } else {
    for (int r = 0; r < 3; ++r) mean[r] /= (double)cnt;
    double cov[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for_neighbours(g, me, rn2, [&](float4, int j) {
      double d[3];
      for (int r = 0; r < 3; ++r) d[r] = pts[3 * (size_t)j + r] - mean[r];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) cov[r][c] += d[r] * d[c];
    });
    smallest_eigenvector(cov, nv);
    const double px = pts[3 * (size_t)i], py = pts[3 * (size_t)i + 1], pz = pts[3 * (size_t)i + 2];
    if ((vx - px) * nv[0] + (vy - py) * nv[1] + (vz - pz) * nv[2] < 0.0) {  // flipNormalTowardsViewpoint
      nv[0] = -nv[0];
      nv[1] = -nv[1];
      nv[2] = -nv[2];
    }
  }
  if (normals)
    for (int r = 0; r < 3; ++r) normals[3 * (size_t)i + r] = nv[r];
  nf[i] = make_float4((float)nv[0], (float)nv[1], (float)nv[2], 0.f);
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
__global__ void __launch_bounds__(FT_THREADS)
    k8_spfh(Grid g, int n, float rf2, const float4* __restrict__ nf, int* __restrict__ counts, int* __restrict__ kcount) {
  __shared__ int hist[FT_DIM][FT_THREADS];
  const int p = blockIdx.x * FT_THREADS + threadIdx.x;
  if (p >= n) return;
  const int tid = threadIdx.x;
  for (int b = 0; b < FT_DIM; ++b) hist[b][tid] = 0;
  const float4 me = g.spts[p];
  const int i = __float_as_int(me.w);
  const float4 ni = nf[i];
  int K = 0;
  constexpr double kPi = 3.14159265358979323846;
  for_neighbours(g, me, rf2, [&](float4 q, int j) {
    ++K;
    float f1, f2, f3;
    if (j == i || !pair_features(me, ni, q, nf[j], f1, f2, f3)) return;
    hist[feature_bin(11.0 * ((double)f1 + kPi) / (2.0 * kPi))][tid] += 1;
    hist[FT_BINS + feature_bin(11.0 * ((double)f2 + 1.0) / 2.0)][tid] += 1;
    hist[2 * FT_BINS + feature_bin(11.0 * ((double)f3 + 1.0) / 2.0)][tid] += 1;
  });
  for (int b = 0; b < FT_DIM; ++b) counts[(size_t)i * FT_DIM + b] = hist[b][tid];
  kcount[i] = K;
}

// ---- FPFH: sum over neighbours j != i at distance > 0 of SPFH_j / |p_j - p_i|^2 (FP64), each 11 bins scaled to 100
__global__ void __launch_bounds__(FT_THREADS)
    k8_fpfh(Grid g, int n, float rf2, const int* __restrict__ counts, const int* __restrict__ kcount,
            float* __restrict__ out) {
  __shared__ double acc[FT_DIM][FT_THREADS];
  const int p = blockIdx.x * FT_THREADS + threadIdx.x;
  if (p >= n) return;
  const int tid = threadIdx.x;
  for (int b = 0; b < FT_DIM; ++b) acc[b][tid] = 0.0;
  const float4 me = g.spts[p];
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

// ---- two-way nearest neighbour over the n_s x n_t matrix of squared L2 distances (difference form, FP32).
// A thread owns NN_ROWS source rows (in registers); a CTA walks one column range in tiles of 2 * NN_PAIRS target
// descriptors staged in shared memory as negated {column c, column c + 1} float2 pairs, so every dimension costs one
// FADD2 (the two differences) and one FFMA2 (the two squares into the two sums) per row.  Row minima stay in the
// thread (ascending columns, strict <: ties keep the lower column) and meet the other column ranges in a packed 64-bit
// atomicMin; column minima go warp -> CTA (shared memory) -> one packed atomicMin per column and CTA.  Key =
// (distance bits << 32) | index: non-negative float bits keep their order and the low word breaks ties.
constexpr int NN_THREADS = 128;
constexpr int NN_ROWS = 2;
constexpr int NN_PAIRS = 32;
constexpr int NN_DP = 34;  // 33 dimensions padded to an even count (the pad is 0 on both sides)
constexpr int NN_COLS_PER_CTA = 2048;

__global__ void __launch_bounds__(NN_THREADS)
    k8_feature_nn(const float* __restrict__ fs, int ns, const float* __restrict__ ft, int nt,
                  unsigned long long* __restrict__ row_key, unsigned long long* __restrict__ col_key) {
  __shared__ __align__(16) float2 tile[NN_PAIRS][NN_DP];
  __shared__ unsigned long long wcol[NN_THREADS / 32][2 * NN_PAIRS];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int row0 = (blockIdx.x * NN_THREADS + tid) * NN_ROWS;  // lane-contiguous rows: lower lane = lower rows
  float a[NN_ROWS][NN_DP];
#pragma unroll
  for (int r = 0; r < NN_ROWS; ++r)
#pragma unroll
    for (int k = 0; k < NN_DP; ++k)
      a[r][k] = (row0 + r < ns && k < FT_DIM) ? fs[(size_t)(row0 + r) * FT_DIM + k] : 0.f;
  unsigned long long best[NN_ROWS];
#pragma unroll
  for (int r = 0; r < NN_ROWS; ++r) best[r] = ~0ull;
  const int c_begin = blockIdx.y * NN_COLS_PER_CTA, c_end = min(nt, c_begin + NN_COLS_PER_CTA);
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

// ---- matcher list (FGR AdvancedMatching): flag[i] for the first part, then one scan places the pairs
// crosscheck: flag[i] = nn_s(nn_t(i)) == i.  one-way: flag[i] = i is nn_s(j) for some j (mark pass below).
__global__ void k8_match_flags(const int* __restrict__ nn_t, int ns, const int* __restrict__ nn_s, int crosscheck,
                               const int* __restrict__ marked, int* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ns) return;
  const int j = nn_t[i];
  flag[i] = crosscheck ? (j >= 0 && nn_s[j] == i) : (marked[i] != 0 && j >= 0);
}

__global__ void k8_match_mark(const int* __restrict__ nn_s, int nt, int* __restrict__ marked) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < nt && nn_s[j] >= 0) marked[nn_s[j]] = 1;
}

// pairs[2k] = source index, pairs[2k + 1] = target index; one-way lists append (nn_s(j), j) for every j after the scan
__global__ void k8_match_place(const int* __restrict__ nn_t, int ns, const int* __restrict__ nn_s, int nt,
                               int crosscheck, const int* __restrict__ flag, const int* __restrict__ pos,
                               int* __restrict__ pairs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < ns && flag[i]) {
    pairs[2 * (size_t)pos[i]] = i;
    pairs[2 * (size_t)pos[i] + 1] = nn_t[i];
  }
  if (!crosscheck && i < nt) {
    const size_t k = (size_t)pos[ns] + i;
    pairs[2 * k] = nn_s[i];
    pairs[2 * k + 1] = i;
  }
}

// ---- tuple test: trial t draws list positions rand31(seed; TUPLE, 0, 3t + k) % ncorr, k = 0, 1, 2, and passes iff
// every source / target edge length ratio of the triangle lies strictly inside (s, 1/s) (FP32, FGR's expression)
__device__ __forceinline__ float len3(const double* __restrict__ P, int a, int b) {
  const float dx = (float)P[3 * (size_t)a] - (float)P[3 * (size_t)b];
  const float dy = (float)P[3 * (size_t)a + 1] - (float)P[3 * (size_t)b + 1];
  const float dz = (float)P[3 * (size_t)a + 2] - (float)P[3 * (size_t)b + 2];
  return __fsqrt_rn(dot3(dx, dy, dz, dx, dy, dz));
}

__global__ void k8_tuple_trials(const double* __restrict__ src, const double* __restrict__ tgt,
                                const int* __restrict__ list, int ncorr, float s, uint64_t seed,
                                unsigned long long t0, int nt, int* __restrict__ pass) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= nt) return;
  const unsigned long long t = t0 + u;
  int r[3];
  for (int k = 0; k < 3; ++k)
    r[k] = (int)(philox_rand31(seed, PSULVSB_DOMAIN_TUPLE, 0u, 3 * t + k) % (uint32_t)ncorr);
  bool ok = true;
  for (int e = 0; e < 3; ++e) {
    const int a = r[e], b = r[(e + 1) % 3];
    const float li = len3(src, list[2 * a], list[2 * b]);
    const float lj = len3(tgt, list[2 * a + 1], list[2 * b + 1]);
    ok = ok && (__fmul_rn(li, s) < lj) && (lj < __fdiv_rn(li, s));
  }
  pass[u] = ok ? 1 : 0;
}

// appends the passing trials of one chunk, in trial order, while fewer than max_tuples have been kept (one CTA)
__global__ void __launch_bounds__(SCAN_THREADS)
    k8_tuple_keep(const int* __restrict__ pass, int nt, unsigned long long t0, const int* __restrict__ list,
                  int ncorr, uint64_t seed, int max_tuples, int* __restrict__ kept, int* __restrict__ out) {
  __shared__ int warp_tot[SCAN_THREADS / 32];
  __shared__ int base;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) base = *kept;
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
        const int r = (int)(philox_rand31(seed, PSULVSB_DOMAIN_TUPLE, 0u, 3 * t + k) % (uint32_t)ncorr);
        out[2 * (3 * (size_t)slot + k)] = list[2 * r];
        out[2 * (3 * (size_t)slot + k) + 1] = list[2 * r + 1];
      }
    }
    __syncthreads();
    if (tid == 0) base = min(max_tuples, base + total);
    __syncthreads();
  }
  if (tid == 0) *kept = base;
}

inline size_t up256(size_t x) { return (x + 255) & ~size_t(255); }

struct FpfhWork {
  int *pbucket, *count, *start, *cursor, *tmp, *counts, *kcount;
  float4 *spts, *nf;
};

size_t fpfh_layout(int n, char* base, FpfhWork* w) {
  const size_t nn = (size_t)(n > 0 ? n : 0), nb = bucket_count(n);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += up256(bytes);
    return p;
  };
  FpfhWork v;
  v.spts = (float4*)take(16 * nn);
  v.nf = (float4*)take(16 * nn);
  v.pbucket = (int*)take(4 * nn);
  v.count = (int*)take(4 * nb);
  v.start = (int*)take(4 * (nb + 1));
  v.cursor = (int*)take(4 * nb);
  v.tmp = (int*)take(4 * nn);
  v.counts = (int*)take(4 * FT_DIM * nn);
  v.kcount = (int*)take(4 * nn);
  if (w) *w = v;
  return off;
}

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

bool radius_ok(double r) { return std::isfinite(r) && r > 0.0; }

inline int blocks(long long n, int t) { return (int)((n + t - 1) / t); }

int run_fpfh(cudaStream_t st, const double* pts, int n, double rn, double rf, const double* viewpoint, void* work,
             double* normals, float* features) {
  if (n == 0) return PSULVSB_OK;
  FpfhWork w;
  fpfh_layout(n, static_cast<char*>(work), &w);
  const unsigned int nb = bucket_count(n);
  const double h = (rn > rf ? rn : rf) * (1.0 + 1e-5);
  Grid g{1.0 / h, nb - 1, w.spts, w.start};
  PSU_CUDA(cudaMemsetAsync(w.count, 0, 4 * (size_t)nb, st));
  k8_grid_count<<<blocks(n, FT_THREADS), FT_THREADS, 0, st>>>(pts, n, g.inv_h, g.mask, w.pbucket, w.count);
  PSU_CHECK_LAUNCH("k8_grid_count");
  k8_scan<<<1, SCAN_THREADS, 0, st>>>(w.count, (int)nb, w.start, w.cursor);
  PSU_CHECK_LAUNCH("k8_scan");
  k8_grid_scatter<<<blocks(n, FT_THREADS), FT_THREADS, 0, st>>>(n, w.pbucket, w.cursor, w.tmp);
  PSU_CHECK_LAUNCH("k8_grid_scatter");
  k8_grid_order<<<blocks(n, FT_THREADS), FT_THREADS, 0, st>>>(pts, n, w.pbucket, w.start, w.tmp, w.spts);
  PSU_CHECK_LAUNCH("k8_grid_order");
  const double vx = viewpoint ? viewpoint[0] : 0.0, vy = viewpoint ? viewpoint[1] : 0.0,
               vz = viewpoint ? viewpoint[2] : 0.0;
  k8_radius_normals<<<blocks(n, FT_THREADS), FT_THREADS, 0, st>>>(g, pts, n, (float)(rn * rn), vx, vy, vz, normals,
                                                                   w.nf);
  PSU_CHECK_LAUNCH("k8_radius_normals");
  k8_spfh<<<blocks(n, FT_THREADS), FT_THREADS, 0, st>>>(g, n, (float)(rf * rf), w.nf, w.counts, w.kcount);
  PSU_CHECK_LAUNCH("k8_spfh");
  k8_fpfh<<<blocks(n, FT_THREADS), FT_THREADS, 0, st>>>(g, n, (float)(rf * rf), w.counts, w.kcount, features);
  PSU_CHECK_LAUNCH("k8_fpfh");
  return PSULVSB_OK;
}

int run_feature_nn(cudaStream_t st, const float* fs, int ns, const float* ft, int nt, int* nn_s2t, int* nn_t2s) {
  if (ns == 0 && nt == 0) return PSULVSB_OK;
  if (ns == 0 || nt == 0) {  // nothing to be near to
    if (ns) PSU_CUDA(cudaMemsetAsync(nn_s2t, 0xFF, 4 * (size_t)ns, st));
    if (nt) PSU_CUDA(cudaMemsetAsync(nn_t2s, 0xFF, 4 * (size_t)nt, st));
    return PSULVSB_OK;
  }
  unsigned long long* keys = nullptr;
  const size_t nk = (size_t)ns + (size_t)nt;
  PSU_CUDA(cudaMallocAsync((void**)&keys, 8 * nk, st));
  int rc = PSULVSB_OK;
  if (cudaMemsetAsync(keys, 0xFF, 8 * nk, st) != cudaSuccess) rc = fail(PSULVSB_ERR_CUDA, "feature nn: memset failed");
  if (!rc) {
    const dim3 grid(blocks(ns, NN_THREADS * NN_ROWS), blocks(nt, NN_COLS_PER_CTA));
    k8_feature_nn<<<grid, NN_THREADS, 0, st>>>(fs, ns, ft, nt, keys, keys + ns);
    if (cudaGetLastError() != cudaSuccess) rc = fail(PSULVSB_ERR_CUDA, "k8_feature_nn launch failed");
  }
  if (!rc) {
    k8_nn_finish<<<blocks(ns, 256), 256, 0, st>>>(keys, ns, nn_s2t);
    k8_nn_finish<<<blocks(nt, 256), 256, 0, st>>>(keys + ns, nt, nn_t2s);
    if (cudaGetLastError() != cudaSuccess) rc = fail(PSULVSB_ERR_CUDA, "k8_nn_finish launch failed");
  }
  cudaFreeAsync(keys, st);
  return rc;
}

constexpr int MAX_TUPLES = 1000;
constexpr int TUPLE_CHUNK = 1 << 20;

// host buffers in: descriptors -> two-way NN -> list -> tuple test; pairs out
int run_match_host(const double* src, int ns, const double* tgt, int nt, const float* fs, const float* ft,
                   int crosscheck, int tuple_test, double tuple_scale, uint64_t seed, int* pairs, long long capacity,
                   long long* n_pairs) {
  *n_pairs = 0;
  cudaStream_t st = nullptr;
  const size_t NS = (size_t)ns, NT = (size_t)nt, NL = NS + NT;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += up256(bytes);
    return o;
  };
  const size_t o_src = take(24 * NS), o_tgt = take(24 * NT), o_fs = take(4 * FT_DIM * NS), o_ft = take(4 * FT_DIM * NT);
  const size_t o_nnt = take(4 * NS), o_nns = take(4 * NT), o_mark = take(4 * NS), o_flag = take(4 * NS),
               o_pos = take(4 * (NS + 1)), o_list = take(8 * NL), o_pass = take(4 * (size_t)TUPLE_CHUNK),
               o_kept = take(4), o_out = take(8 * 3 * (size_t)MAX_TUPLES);
  DevBuf buf;
  if (int rc = buf.alloc(off, "psulvsb_match_host")) return rc;
  char* b = static_cast<char*>(buf.p);
  double* d_src = (double*)(b + o_src);
  double* d_tgt = (double*)(b + o_tgt);
  float* d_fs = (float*)(b + o_fs);
  float* d_ft = (float*)(b + o_ft);
  int *nn_t = (int*)(b + o_nnt), *nn_s = (int*)(b + o_nns), *mark = (int*)(b + o_mark), *flag = (int*)(b + o_flag),
      *pos = (int*)(b + o_pos), *list = (int*)(b + o_list), *pass = (int*)(b + o_pass), *kept = (int*)(b + o_kept),
      *out = (int*)(b + o_out);
  PSU_CUDA(cudaMemcpyAsync(d_src, src, 24 * NS, cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaMemcpyAsync(d_tgt, tgt, 24 * NT, cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaMemcpyAsync(d_fs, fs, 4 * FT_DIM * NS, cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaMemcpyAsync(d_ft, ft, 4 * FT_DIM * NT, cudaMemcpyHostToDevice, st));
  if (int rc = run_feature_nn(st, d_fs, ns, d_ft, nt, nn_t, nn_s)) return rc;
  PSU_CUDA(cudaMemsetAsync(mark, 0, 4 * NS, st));
  k8_match_mark<<<blocks(nt, 256), 256, 0, st>>>(nn_s, nt, mark);
  PSU_CHECK_LAUNCH("k8_match_mark");
  k8_match_flags<<<blocks(ns, 256), 256, 0, st>>>(nn_t, ns, nn_s, crosscheck, mark, flag);
  PSU_CHECK_LAUNCH("k8_match_flags");
  k8_scan<<<1, SCAN_THREADS, 0, st>>>(flag, ns, pos, nullptr);
  PSU_CHECK_LAUNCH("k8_scan");
  const int nplace = ns > nt ? ns : nt;
  k8_match_place<<<blocks(nplace, 256), 256, 0, st>>>(nn_t, ns, nn_s, nt, crosscheck, flag, pos, list);
  PSU_CHECK_LAUNCH("k8_match_place");
  int first = 0;
  PSU_CUDA(cudaMemcpyAsync(&first, pos + ns, 4, cudaMemcpyDeviceToHost, st));
  PSU_CUDA(cudaStreamSynchronize(st));
  const long long ncorr = (long long)first + (crosscheck ? 0 : nt);
  const int* result = list;
  long long count = ncorr;
  if (tuple_test) {
    count = 0;
    PSU_CUDA(cudaMemsetAsync(kept, 0, 4, st));
    const unsigned long long trials = 100ull * (unsigned long long)ncorr;
    int got = 0;
    for (unsigned long long t0 = 0; t0 < trials && got < MAX_TUPLES; t0 += TUPLE_CHUNK) {
      const int chunk = (int)(trials - t0 < (unsigned long long)TUPLE_CHUNK ? trials - t0 : TUPLE_CHUNK);
      k8_tuple_trials<<<blocks(chunk, 256), 256, 0, st>>>(d_src, d_tgt, list, (int)ncorr, (float)tuple_scale, seed, t0,
                                                          chunk, pass);
      PSU_CHECK_LAUNCH("k8_tuple_trials");
      k8_tuple_keep<<<1, SCAN_THREADS, 0, st>>>(pass, chunk, t0, list, (int)ncorr, seed, MAX_TUPLES, kept, out);
      PSU_CHECK_LAUNCH("k8_tuple_keep");
      PSU_CUDA(cudaMemcpyAsync(&got, kept, 4, cudaMemcpyDeviceToHost, st));
      PSU_CUDA(cudaStreamSynchronize(st));
    }
    count = 3ll * got;
    result = out;
  }
  *n_pairs = count;
  if (count > capacity)
    return fail(PSULVSB_ERR_CAPACITY, "psulvsb_match_host: " + std::to_string(count) + " pairs, capacity " +
                                          std::to_string(capacity));
  if (count) PSU_CUDA(cudaMemcpyAsync(pairs, result, 8 * (size_t)count, cudaMemcpyDeviceToHost, st));
  PSU_CUDA(cudaStreamSynchronize(st));
  return PSULVSB_OK;
}

}  // namespace

}  // namespace psulvsb

using psulvsb::fail;

extern "C" {

unsigned long long psulvsb_fpfh_workspace_bytes(int n) {
  return n < 0 ? 0ull : (unsigned long long)psulvsb::fpfh_layout(n, nullptr, nullptr);
}

int psulvsb_fpfh(void* stream, const double* d_pts, int n, double normal_radius, double feature_radius,
                 const double viewpoint[3], void* d_work, double* d_normals, float* d_features) {
  if (n < 0 || !psulvsb::radius_ok(normal_radius) || !psulvsb::radius_ok(feature_radius) ||
      (n > 0 && (!d_pts || !d_work || !d_features)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_fpfh: bad argument (radii must be finite and > 0)");
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_fpfh((cudaStream_t)stream, d_pts, n, normal_radius, feature_radius, viewpoint, d_work, d_normals,
                           d_features);
}

int psulvsb_fpfh_host(const double* pts, int n, double normal_radius, double feature_radius, const double viewpoint[3],
                      double* normals, float* features) {
  if (n < 0 || !psulvsb::radius_ok(normal_radius) || !psulvsb::radius_ok(feature_radius) ||
      (n > 0 && (!pts || !features)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_fpfh_host: bad argument (radii must be finite and > 0)");
  if (int rc = psulvsb::need_device()) return rc;
  if (n == 0) return PSULVSB_OK;
  const size_t nn = (size_t)n, o_f = psulvsb::up256(24 * nn), o_n = o_f + psulvsb::up256(4 * 33 * nn),
               o_w = o_n + psulvsb::up256(24 * nn);
  psulvsb::DevBuf buf;
  if (int rc = buf.alloc(o_w + psulvsb_fpfh_workspace_bytes(n), "psulvsb_fpfh_host")) return rc;
  char* b = static_cast<char*>(buf.p);
  PSU_CUDA(cudaMemcpy(b, pts, 24 * nn, cudaMemcpyHostToDevice));
  if (int rc = psulvsb::run_fpfh(nullptr, (double*)b, n, normal_radius, feature_radius, viewpoint, b + o_w,
                                 normals ? (double*)(b + o_n) : nullptr, (float*)(b + o_f)))
    return rc;
  PSU_CUDA(cudaMemcpy(features, b + o_f, 4 * 33 * nn, cudaMemcpyDeviceToHost));
  if (normals) PSU_CUDA(cudaMemcpy(normals, b + o_n, 24 * nn, cudaMemcpyDeviceToHost));
  return PSULVSB_OK;
}

int psulvsb_feature_nn(void* stream, const float* d_fs, int n_src, const float* d_ft, int n_tgt, int* d_nn_src_to_tgt,
                       int* d_nn_tgt_to_src) {
  if (n_src < 0 || n_tgt < 0 || (n_src > 0 && (!d_fs || !d_nn_src_to_tgt)) || (n_tgt > 0 && (!d_ft || !d_nn_tgt_to_src)))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_feature_nn: bad argument");
  if (int rc = psulvsb::need_device()) return rc;
  return psulvsb::run_feature_nn((cudaStream_t)stream, d_fs, n_src, d_ft, n_tgt, d_nn_src_to_tgt, d_nn_tgt_to_src);
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
  return psulvsb::run_match_host(src_pts, n_src, tgt_pts, n_tgt, fs, ft, crosscheck, tuple_test, tuple_scale, seed,
                                 pairs, capacity, n_pairs);
}

}  // extern "C"
