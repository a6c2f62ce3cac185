// ft_voxel.cuh -- the voxel-grid filter's pipeline (Open3D's PointCloud::VoxelDownSample), shared by the plain filter
// (k8_voxel.cu) and the colour-carrying one (k8_voxel_colors.cu), on the FPFH stage's batch table and hashed grid
// (ft_batch.cuh, grid.cuh).  DESIGN.md section 10, "Voxel downsampling", is the specification;
// tests/voxel_restatement.py restates it in numpy.
//
// Per cloud: lo = the exact minimum of the finite points per coordinate, origin = lo - v * 0.5, and the cell of a
// finite point is floor((p - origin) / v) per coordinate in FP64, saturated to int64.  Cells hash into the cloud's
// bucket_count(n) buckets; each bucket's members are ranked by index, so a walk over a bucket meets them in ascending
// index order.  A point is its voxel's representative iff no earlier member of its bucket has its cell; the
// representatives take the output columns in ascending index order, and each writes the mean of its voxel's members,
// summed in ascending index order.  Two points share a voxel iff their three cells are equal: the hash only groups.
#pragma once

#include <cuda_runtime.h>

#include <cmath>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "ft_batch.cuh"
#include "grid.cuh"

namespace psulvsb {

namespace {

struct Cell {
  long long x, y, z;
};

__device__ __forceinline__ bool same_cell(const Cell& a, const Cell& b) { return a.x == b.x && a.y == b.y && a.z == b.z; }

// the order-preserving unsigned image of a double (not NaN), complemented: the minimum of the doubles is the maximum of
// the keys, so a zeroed slot is the identity and one memset clears the bounds together with the bucket counts
__device__ __forceinline__ unsigned long long min_key(double x) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return ~((b >> 63) ? ~b : b | 0x8000000000000000ull);
}

__device__ __forceinline__ double from_min_key(unsigned long long k) {
  const unsigned long long b = ~k;
  return __longlong_as_double((long long)((b >> 63) ? b & 0x7FFFFFFFFFFFFFFFull : ~b));
}

__device__ __forceinline__ bool finite3(double x, double y, double z) { return isfinite(x) && isfinite(y) && isfinite(z); }

// one subtraction, one division, floor; the conversion saturates (cvt.rzi.s64.f64), so a cloud whose extent over v
// exceeds the int64 range puts its far points in the last cell instead of failing
__device__ __forceinline__ long long cell1(double p, double origin, double v) { return (long long)floor((p - origin) / v); }

// ---- per-cloud bounds: each CTA reduces its tile's finite points, then one atomicMax per coordinate (min is exact, so
// the result does not depend on the order of the atomics)
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS)
    k8_voxel_bounds(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one,
                    const int* __restrict__ tile_first, int B, unsigned long long* __restrict__ lo) {
  __shared__ unsigned long long part[3][FT_THREADS / 32];
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int i = first + threadIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned long long k[3] = {0ull, 0ull, 0ull};
  if (i < cl.n) {
    const double* p = cl.pts + 3 * (size_t)i;
    const double x = p[0], y = p[1], z = p[2];
    if (finite3(x, y, z)) {
      k[0] = min_key(x);
      k[1] = min_key(y);
      k[2] = min_key(z);
    }
  }
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) k[r] = max(k[r], __shfl_xor_sync(0xffffffffu, k[r], o));
    if (lane == 0) part[r][wid] = k[r];
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    unsigned long long m = 0ull;
    for (int w = 0; w < FT_THREADS / 32; ++w) m = max(m, part[threadIdx.x][w]);
    if (m) atomicMax(lo + 3 * ci + threadIdx.x, m);
  }
}

// ---- cell and bucket of every point; a non-finite point gets bucket -1 and stays out of the grid
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS)
    k8_voxel_count(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one,
                   const int* __restrict__ tile_first, int B, double v, const unsigned long long* __restrict__ lo,
                   int* __restrict__ pbucket, Cell* __restrict__ pcell, int* __restrict__ count) {
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int i = first + threadIdx.x;
  if (i >= cl.n) return;
  const double* p = cl.pts + 3 * (size_t)i;
  const double x = p[0], y = p[1], z = p[2];
  const size_t o = (size_t)cl.p0 + i;
  if (!finite3(x, y, z)) {
    pbucket[o] = -1;
    return;
  }
  const double h = v * 0.5;
  const Cell c{cell1(x, from_min_key(lo[3 * ci]) - h, v), cell1(y, from_min_key(lo[3 * ci + 1]) - h, v),
               cell1(z, from_min_key(lo[3 * ci + 2]) - h, v)};
  const int b = cl.b0 + (int)bucket_of(c.x, c.y, c.z, cl.mask);
  pbucket[o] = b;
  pcell[o] = c;
  atomicAdd(count + b, 1);
}

// ---- rank each member of a bucket by index (the scatter's order depends on timing); per sorted slot the index in the
// cloud and the cell, per point its sorted position.  Slots past the cloud's grid belong to points left out of it.
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS)
    k8_voxel_order(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one,
                   const int* __restrict__ tile_first, int B, const int* __restrict__ pbucket,
                   const int* __restrict__ start, const int* __restrict__ tmp, const Cell* __restrict__ pcell,
                   int* __restrict__ spos, int* __restrict__ sidx, Cell* __restrict__ scell) {
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int l = first + threadIdx.x;
  if (l >= cl.n) return;
  const int s = cl.p0 + l;
  if (s >= start[cl.b0 + ci + cl.mask + 1]) return;
  const int i = tmp[s];
  const int b = pbucket[i] + ci, s0 = start[b], s1 = start[b + 1];
  int rank = 0;
  for (int q = s0; q < s1; ++q) rank += tmp[q] < i;
  const int d = s0 + rank;
  sidx[d] = i - cl.p0;
  scell[d] = pcell[i];
  spos[i] = d;
}

// ---- representatives: point i is one iff no earlier member of its bucket has its cell; tile_count[tile] = how many
// the tile holds
template <bool kBatch>
__global__ void __launch_bounds__(FT_THREADS)
    k8_voxel_first(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one,
                   const int* __restrict__ tile_first, int B, const int* __restrict__ pbucket,
                   const int* __restrict__ start, const int* __restrict__ spos, const Cell* __restrict__ scell,
                   unsigned char* __restrict__ rep, int* __restrict__ tile_count) {
  __shared__ int warp_n[FT_THREADS / 32];
  int ci, first;
  const FtCloud& cl = cloud_tile<kBatch>(clouds, one, tile_first, B, ci, first);
  const int i = first + threadIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  bool r = false;
  if (i < cl.n) {
    const size_t o = (size_t)cl.p0 + i;
    const int b = pbucket[o];
    if (b >= 0) {
      const int s = spos[o];
      const Cell c = scell[s];
      r = true;
      for (int t = start[b + ci]; t < s && r; ++t) r = !same_cell(scell[t], c);
    }
    rep[o] = r;
  }
  const unsigned int bal = __ballot_sync(0xffffffffu, r);
  if (lane == 0) warp_n[wid] = __popc(bal);
  __syncthreads();
  if (threadIdx.x == 0) {
    int n = 0;
    for (int w = 0; w < FT_THREADS / 32; ++w) n += warp_n[w];
    tile_count[blockIdx.x] = n;
  }
}

// ---- one CTA per cloud: exclusive scan of its tiles' counts at tile_start[tile_first[c] + c ..]; the total is the
// cloud's voxel count
template <bool kBatch>
__global__ void __launch_bounds__(SCAN_THREADS)
    k8_voxel_scan(const FtCloud* __restrict__ clouds, __grid_constant__ const FtCloud one,
                  const int* __restrict__ tile_first, const int* __restrict__ tile_count, int* __restrict__ tile_start,
                  int* __restrict__ counts) {
  const FtCloud& cl = kBatch ? clouds[blockIdx.x] : one;
  if (cl.n == 0) {
    if (threadIdx.x == 0) counts[blockIdx.x] = 0;
    return;
  }
  const int t0 = kBatch ? tile_first[blockIdx.x] : 0, m = (cl.n + FT_THREADS - 1) / FT_THREADS;
  int* st = tile_start + t0 + blockIdx.x;
  cta_scan(tile_count + t0, m, st, nullptr, 0);
  if (threadIdx.x == 0) counts[blockIdx.x] = st[m];
}

struct VoxelWork {
  FtCloud* cloud;  // [B], followed by tile_first [B + 1]: one copy uploads both
  int* tile_first;
  size_t table_bytes;
  unsigned long long* lo;  // [3 B] bound keys, followed by count [nb]: one memset clears both
  int* count;
  size_t zero_bytes;
  int *start, *cursor;                   // [nb + B], [nb]
  int *pbucket, *tmp, *spos, *sidx;      // [n]
  Cell *pcell, *scell;                   // [n]: per point, per sorted slot
  unsigned char* rep;                    // [n]
  int *tile_count, *tile_start;          // [tiles], [tiles + B]
};

size_t voxel_layout(const FpfhSizes& z, char* base, VoxelWork* w) {
  const size_t nn = (size_t)z.n, nb = (size_t)z.nb, B = (size_t)z.B, tiles = (size_t)z.tiles;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += up256(bytes);
    return p;
  };
  VoxelWork v;
  v.table_bytes = sizeof(FtCloud) * B + 4 * (B + 1);
  v.cloud = (FtCloud*)take(v.table_bytes);
  v.tile_first = (int*)((char*)v.cloud + sizeof(FtCloud) * B);
  v.zero_bytes = 8 * 3 * B + 4 * nb;
  v.lo = (unsigned long long*)take(v.zero_bytes);
  v.count = (int*)(v.lo + 3 * B);
  v.start = (int*)take(4 * (nb + B));
  v.cursor = (int*)take(4 * nb);
  v.pbucket = (int*)take(4 * nn);
  v.tmp = (int*)take(4 * nn);
  v.spos = (int*)take(4 * nn);
  v.sidx = (int*)take(4 * nn);
  v.pcell = (Cell*)take(sizeof(Cell) * nn);
  v.scell = (Cell*)take(sizeof(Cell) * nn);
  v.rep = (unsigned char*)take(nn);
  v.tile_count = (int*)take(4 * tiles);
  v.tile_start = (int*)take(4 * (tiles + B));
  if (w) *w = v;
  return off;
}

bool voxel_ok(double v) { return std::isfinite(v) && v > 0.0; }

// the seven passes ahead of the mean
template <bool kBatch>
void launch_voxel_grid(cudaStream_t st, const VoxelWork& w, const FtCloud& one, int B, int tiles, int n, double v,
                       int* counts) {
  k8_voxel_bounds<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, w.lo);
  k8_voxel_count<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, v, w.lo, w.pbucket, w.pcell,
                                                       w.count);
  k8_cloud_scan<kBatch><<<B, SCAN_THREADS, 0, st>>>(w.cloud, one, w.count, w.start, w.cursor);
  k8_grid_scatter<<<blocks(n, GRID_THREADS), GRID_THREADS, 0, st>>>(n, w.pbucket, w.cursor, w.tmp);
  k8_voxel_order<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, w.pbucket, w.start, w.tmp,
                                                       w.pcell, w.spos, w.sidx, w.scell);
  k8_voxel_first<kBatch><<<tiles, FT_THREADS, 0, st>>>(w.cloud, one, w.tile_first, B, w.pbucket, w.start, w.spos,
                                                       w.scell, w.rep, w.tile_count);
  k8_voxel_scan<kBatch><<<B, SCAN_THREADS, 0, st>>>(w.cloud, one, w.tile_first, w.tile_count, w.tile_start, counts);
}

// the batch on the device (clouds checked, B >= 1): one upload of the cloud table (batches only), one memset, the seven
// passes ahead of the mean over all clouds, then mean(std::bool_constant<kBatch>, w, one, tiles) launches the mean
// pass; every count is written on the device
template <class Mean>
int run_voxel_passes(cudaStream_t st, const psulvsb_fpfh_cloud_t* clouds, int B, double v, void* work, int* counts,
                     Mean mean) {
  const FpfhSizes z = fpfh_sizes(clouds, B);
  if (z.tiles == 0) {
    PSU_CUDA(cudaMemsetAsync(counts, 0, 4 * (size_t)B, st));
    return PSULVSB_OK;
  }
  VoxelWork w;
  voxel_layout(z, static_cast<char*>(work), &w);
  std::vector<char> table(w.table_bytes);
  FtCloud* hc = reinterpret_cast<FtCloud*>(table.data());
  int* tile_first = reinterpret_cast<int*>(table.data() + sizeof(FtCloud) * (size_t)B);
  tile_first[0] = 0;
  long long p0 = 0, b0 = 0;
  for (int c = 0; c < B; ++c) {
    const psulvsb_fpfh_cloud_t& q = clouds[c];
    FtCloud& h = hc[c];
    const unsigned int nb = q.n > 0 ? bucket_count(q.n) : 0u;
    h = FtCloud{};
    h.pts = q.pts;
    h.n = q.n;
    h.p0 = (int)p0;
    h.b0 = (int)b0;
    h.mask = nb - 1;
    p0 += q.n;
    b0 += nb;
    tile_first[c + 1] = tile_first[c] + blocks(q.n, FT_THREADS);
  }
  if (B > 1) PSU_CUDA(cudaMemcpyAsync(w.cloud, table.data(), table.size(), cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaMemsetAsync(w.lo, 0, w.zero_bytes, st));
  const int tiles = (int)z.tiles, n = (int)z.n;
  if (B == 1) {
    launch_voxel_grid<false>(st, w, hc[0], 1, tiles, n, v, counts);
    if (int rc = mean(std::false_type{}, w, hc[0], tiles)) return rc;
  } else {
    launch_voxel_grid<true>(st, w, hc[0], B, tiles, n, v, counts);
    if (int rc = mean(std::true_type{}, w, hc[0], tiles)) return rc;
  }
  PSU_CHECK_LAUNCH("k8_voxel_mean");
  return PSULVSB_OK;
}

}  // namespace

}  // namespace psulvsb
