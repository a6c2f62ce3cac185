// k3_rotation.cu -- stage 3: GNC-TLS rotation (thread-block cluster per hypothesis) and batched
// closed-form Kabsch (one warp per hypothesis).
//
// Reference: GNCTLSRotationSolver::solveForRotation (registration.cc:1563-1692) around
// teaser::utils::svdRot (utils.h:121-136).  All arithmetic is FP64: the rotation feeds
// discontinuous decisions downstream (w >= 0.5 inlier test, max-stabbing translation), so FP32
// here would break the 1e-5 parity bar (DESIGN.md "Why FP64 in stage 3").
//
// One GNC iteration is ONE pass over the K line vectors: with R_i known every thread computes
// r^2 = |tv - R_i sv|^2, adds w_{i-1} r^2 to the cost, updates the weight in closed form and
// accumulates H_{i+1} += w_i sv tv^T; the partial sums are reduced warp -> CTA -> cluster (distributed shared
// memory) in a fixed order (deterministic), and thread 0 of every CTA turns H into R_{i+1} (Newton step on SO(3)
// from R_i, 3x3 Jacobi SVD when it declines), decides about convergence and publishes the next pass's constants
// -- two CTA barriers per iteration.
//
// Layout.  A CTA's contiguous slice of the line vectors is cut into one contiguous SEGMENT PER WARP; a warp walks
// its segment 64 positions at a time (two coalesced groups in flight per lane).  The first positions of every
// segment live in the warp's share of shared memory (sv, tv, slot: 56 bytes), the rest in a coalesced SoA scratch in
// HBM/L2 (GncJob::lv, GncJob::weights), and only what exceeds that too is re-formed from the points each pass.  The
// cluster size (1, 2, 4 or 8 CTAs per hypothesis) is chosen by the launcher from the batch size: few registrations
// -> 8 SMs each (latency), many -> one SM each (throughput).
//
// Sleeping line vectors.  Once mu has grown, most outliers sit at weight 0 and stay there: w = 0 iff
// r >= sqrt(th1), th1 only shrinks (mu grows), and a rotation change moves a residual by at most
// |R_new - R_old|_2 |sv|.  A line vector found with w = 0 and margin m = (r - sqrt(th1)) / |sv| therefore keeps
// w = 0 -- contributing nothing to the cost (its previous weight is 0) nor to H -- until the accumulated
// drift sum |R_{i+1} - R_i|_F has grown by m.  Its slot then stores -(drift + m) ("asleep until the drift reaches
// this"); while the remaining margin is at least 0.005 rad (a DEEP sleeper) the pass skips it exactly; nothing is
// approximated.  When enough of a CTA's positions sleep deeply the next pass is ARMED: every warp drops its deep
// sleepers and moves the others down inside its own segment, in order, as part of the pass (a warp vote gives the
// new positions; no barrier, no second sweep, and the survivors migrate into the shared-memory part of the segment
// as it shrinks; their original indices travel in GncJob::perm for the epilogue).  Parking overwrites the parked
// line vectors; the cluster keeps the smallest wake-up drift among them, and if the drift ever reaches it (rare:
// the parking margin is consumed only by a late jump of the rotation) the solve is repeated without sleeping.
// On cfg-A (K = 22 000, 95 % outliers) 60 % of the line-vector evaluations of a solve disappear.
// FP64 with explicit fma(): reduction order already differs from a sequential CPU sum, so fusing
// adds no new class of deviation; the discrete decisions (r^2 vs th1/th2, w >= 0.5) are unaffected
// except within an ulp of their thresholds.
#include <cooperative_groups.h>
#include <algorithm>
#include <cstdlib>
#include <cuda_runtime.h>
#include <type_traits>

#include "common.cuh"
#include "engine.cuh"
#include "svd3.cuh"

namespace cg = cooperative_groups;

namespace psulvsb {

namespace {

// threads per CTA is a template parameter T: 256 (two CTAs per SM, so that one hypothesis' serial rotation update
// overlaps another's pass) for clustered launches, 512 (one CTA per SM, twice the shared-memory cache) when
// every hypothesis runs on a single CTA (large batches)
constexpr int GNC_CTAS_PER_SM = 2;

__device__ __forceinline__ void load_lv(const double* __restrict__ src, const double* __restrict__ dst, uint2 e,
                                        double inv_scale, double sv[3], double tv[3]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    sv[r] = src[3 * (size_t)e.y + r] - src[3 * (size_t)e.x + r];
    // pruned_dst_tims_ *= (1 / solution_.scale)   (registration.cc:1102)
    tv[r] = (dst[3 * (size_t)e.y + r] - dst[3 * (size_t)e.x + r]) * inv_scale;
  }
}

// the same from 64-byte point records: six 16-byte read-only loads, four sectors
__device__ __forceinline__ void load_lv8(const double* __restrict__ pts8, uint2 e, double inv_scale, double sv[3],
                                         double tv[3]) {
  const double2* pa = reinterpret_cast<const double2*>(pts8 + 8 * (size_t)e.x);
  const double2* pb = reinterpret_cast<const double2*>(pts8 + 8 * (size_t)e.y);
  const double2 a0 = __ldg(pa), a1 = __ldg(pa + 1), a2 = __ldg(pa + 2);
  const double2 b0 = __ldg(pb), b1 = __ldg(pb + 1), b2 = __ldg(pb + 2);
  sv[0] = b0.x - a0.x;
  sv[1] = b0.y - a0.y;
  sv[2] = b1.x - a1.x;
  tv[0] = (b1.y - a1.y) * inv_scale;  // pruned_dst_tims_ *= (1 / solution_.scale)   (registration.cc:1102)
  tv[1] = (b2.x - a2.x) * inv_scale;
  tv[2] = (b2.y - a2.y) * inv_scale;
}

// ------------------------------------------------------------------------------------------
// GNC-TLS, one cluster of NC CTAs per registration.  See the header comment for the layout.
// ------------------------------------------------------------------------------------------
constexpr int GNC_MAX_WARPS = 16;  // T <= 512
constexpr int GNC_NRED = 16;
// slots of the per-iteration reduction: 0..8 = H (row-major), then
constexpr int RED_COST = 9;   // sum w_{i-1} r_i^2
constexpr int RED_DEEP = 10;  // deep sleepers left inside the warps' ranges
constexpr int RED_LEFT = 11;  // positions left inside the warps' ranges
constexpr int RED_MAX = 15;   // reduced with max: max r^2 (first pass) / -(smallest wake-up drift parked in this pass)
constexpr double GNC_DEEP_MARGIN_DEFAULT = 0.005;  // remaining margin (rad) from which a sleeping line vector is parked
constexpr int GNC_PF_STEPS = 1;   // look-ahead (double-steps) of the L2 prefetch in the streamed pass (1, 2, 4 measured equal)
constexpr int GNC_PARK_PCT = 45;  // share (%) of a CTA's positions that must sleep deeply before a pass is armed

// what thread 0 decides between two passes; everyone reads it after ONE barrier
struct GncCtl {
  double th1, th2, sqrt_wnum, mu, drift;
  float sqrt_th1_up;
  int stop;     // 1: the loop ends (converged / last iteration), 2: degenerate mu at the first iteration
  int armed;    // the next pass parks its deep sleepers
  int reopen;   // a parked line vector may wake up: all parked ones return to the ranges
};

struct GncSmem {
  double warp_part[GNC_MAX_WARPS][GNC_NRED];
  double part[2][GNC_NRED];  // this CTA's partial results, double-buffered by reduction parity (peers read them)
  double total[GNC_NRED];
  double R[9];   // row-major current rotation
  double Vw[9];  // Jacobi warm start (right singular vectors of the previous solve), row-major
  GncCtl ctl;
  // thread 0's loop state
  double drift;     // sum of |R_new - R_old|_F over the rotation updates so far
  double min_wake;  // smallest wake-up drift among the parked line vectors (cluster-wide)
  double mu, prev_cost, cost;
  // diagnostics of thread 0 (GncJob::prof): pass / rotation-update cycles, positions evaluated, armed passes
  long long t_stream, t_svd, sum_act, t_prologue, t_start;
  int n_armed, first_armed;
};

// 1 / sqrt(x) for a finite x > 0 (x = 0 gives inf, selected away by the caller): the 20-bit seed of MUFU.RSQ64H and
// two Newton steps with a correction term -- within an ulp of the correctly rounded value, without the special-case
// handling of rsqrt() (the weight it feeds is formed differently from the reference's sqrt(a / r^2) anyway)
__device__ __forceinline__ double rsqrt_pos(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double hx = 0.5 * x;
  double e = fma(-hx * y, y, 0.5);  // 0.5 - 0.5 x y^2
  y = fma(y, e, y);
  e = fma(-hx * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-hx * y, y, 0.5);
  return fma(y, e, y);
}

__device__ __forceinline__ double residual2(const double R[9], const double sv[3], const double tv[3]) {
  const double d0 = fma(-R[2], sv[2], fma(-R[1], sv[1], fma(-R[0], sv[0], tv[0])));
  const double d1 = fma(-R[5], sv[2], fma(-R[4], sv[1], fma(-R[3], sv[0], tv[1])));
  const double d2 = fma(-R[8], sv[2], fma(-R[7], sv[1], fma(-R[6], sv[0], tv[2])));
  return fma(d2, d2, fma(d1, d1, d0 * d0));
}

// H = sm->total[0..8] -> sm->R, warm-started from / updating sm->Vw.  Out of line on purpose: one thread
// runs it, and inlining its ~600 instructions would set the register budget of the streaming loops
// around it; its operands travel through shared memory, not through local-memory arrays.
__device__ __noinline__ void svd_from_smem(GncSmem* sm) {
  double H[3][3], R[3][3], V[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      H[r][c] = sm->total[r * 3 + c];
      V[r][c] = sm->Vw[r * 3 + c];
    }
  kabsch_rotation(H, R, V);
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      sm->R[r * 3 + c] = R[r][c];
      sm->Vw[r * 3 + c] = V[r][c];
    }
}

// Inside the GNC loop: Newton update from the previous iteration's rotation, Jacobi SVD when it declines.
__device__ __noinline__ void rotation_from_smem(GncSmem* sm) {
  double H[3][3], R[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      H[r][c] = sm->total[r * 3 + c];
      R[r][c] = sm->R[r * 3 + c];
    }
  double d2 = 0.0;
  if (rotation_newton(H, R)) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double d = R[r][c] - sm->R[r * 3 + c];
        d2 = fma(d, d, d2);
        sm->R[r * 3 + c] = R[r][c];
      }
  } else {
    svd_from_smem(sm);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double d = R[r][c] - sm->R[r * 3 + c];
        d2 = fma(d, d, d2);
      }
  }
  // |R_new - R_old|_2 <= |.|_F, rounded up: every residual moved by at most this much times |sv|
  sm->drift += sqrt(d2) * (1.0 + 1e-9) + 1e-15;
}

// ------------------------------------------------------------------------------------------
// Tiny problems (K <= GNC_SERIAL_MAX line vectors): one thread replays GNCTLSRotationSolver::solveForRotation
// (registration.cc:1563-1692) with the reference's sequential sums and operation order (this file is built with
// -fmad=false; no fma() below), the two-sided Jacobi of svd3.cuh standing in for Eigen's.  A basic subset of ONE line
// vector makes H = w x y^T rank 1, where R = V U^T is decided by how the algorithm completes the null space from
// 1-ulp entries: only the same arithmetic reproduces the oracle's R there (and with it the rest of the run).
// ------------------------------------------------------------------------------------------
constexpr int GNC_SERIAL_MAX = 32;

__device__ __noinline__ void gnc_tls_serial(const GncJob& job_g) {
  const GncJob job = job_g;
  const int K = (int)job.K;
  double sv[GNC_SERIAL_MAX][3], tv[GNC_SERIAL_MAX][3], w[GNC_SERIAL_MAX], res[GNC_SERIAL_MAX];
  for (int k = 0; k < K; ++k) {
    load_lv(job.src, job.dst, job.edges[k], job.inv_scale, sv[k], tv[k]);
    w[k] = 1.0;
  }
  double nb2 = job.noise_bound * job.noise_bound;
  if (nb2 < 1e-16) nb2 = 1e-2;  // registration.cc:1592-1595
  double mu = 1.0, prev_cost = INFINITY, cost = INFINITY;
  double R[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  bool use_init = job.use_init != 0;
  int it_done = 0;
  for (int it = 0; it < job.max_iterations; ++it) {
    it_done = it + 1;
    if (use_init) {  // registration.cc:1617-1621
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[r][c] = job.R_init[c * 3 + r];
      use_init = false;
    } else {  // svdRot, utils.h:121-136
      double H[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
      for (int k = 0; k < K; ++k)
        for (int r = 0; r < 3; ++r) {
          const double xw = sv[k][r] * w[k];
          for (int c = 0; c < 3; ++c) H[r][c] += xw * tv[k][c];
        }
      Svd3 d;
      svd3_two_sided(H, d);
      rotation_from_svd(d, R);
    }
    for (int k = 0; k < K; ++k) {
      const double d0 = tv[k][0] - ((R[0][0] * sv[k][0] + R[0][1] * sv[k][1]) + R[0][2] * sv[k][2]);
      const double d1 = tv[k][1] - ((R[1][0] * sv[k][0] + R[1][1] * sv[k][1]) + R[1][2] * sv[k][2]);
      const double d2 = tv[k][2] - ((R[2][0] * sv[k][0] + R[2][1] * sv[k][1]) + R[2][2] * sv[k][2]);
      res[k] = (d0 * d0 + d1 * d1) + d2 * d2;
    }
    if (it == 0) {  // registration.cc:1628-1639
      double max_residual = K > 0 ? res[0] : 0.0;
      for (int k = 1; k < K; ++k) max_residual = (max_residual < res[k]) ? res[k] : max_residual;
      mu = 1 / (2 * max_residual / nb2 - 1);
      if (mu <= 0) break;
    }
    const double th1 = (mu + 1) / mu * nb2, th2 = mu / (mu + 1) * nb2;
    cost = 0;
    for (int k = 0; k < K; ++k) {
      cost += w[k] * res[k];
      if (res[k] >= th1)
        w[k] = 0;
      else if (res[k] <= th2)
        w[k] = 1;
      else
        w[k] = sqrt(nb2 * mu * (mu + 1) / res[k]) - mu;
    }
    const double cost_diff = fabs(cost - prev_cost);
    mu = mu * job.gnc_factor;
    prev_cost = cost;
    if (cost_diff < job.cost_threshold) break;
  }
  int gf = 0;
  for (int k = 0; k < K; ++k) gf += (w[k] >= 0.5) ? 1 : 0;
  const bool all_in = gf <= 10;  // registration.cc:1685-1690
  for (int k = 0; k < K; ++k) {
    const bool in = all_in || w[k] >= 0.5;
    if (job.inliers) job.inliers[k] = in ? 1 : 0;
    if (in && job.point_flags) {
      const uint2 e = job.edges[k];
      job.point_flags[e.x] = 1;
      job.point_flags[e.y] = 1;
    }
  }
  if (job.R_out)
    for (int c = 0; c < 3; ++c)
      for (int r = 0; r < 3; ++r) job.R_out[c * 3 + r] = R[r][c];
  if (job.info) {
    job.info[0] = it_done;
    job.info[1] = all_in ? K : gf;
    job.info[2] = 0;
    job.info[3] = 0;
  }
  if (job.cost) job.cost[0] = cost;
}

// one CTA per job; jobs above GNC_SERIAL_MAX line vectors belong to gnc_tls_kernel
__global__ void __launch_bounds__(128) gnc_tls_small_kernel(const GncJob* __restrict__ jobs) {
  const GncJob& job = jobs[blockIdx.x];
  if (threadIdx.x == 0 && job.grid_bar) *job.grid_bar = 0u;  // (grid mode of gnc_tls_kernel, launched after this one)
  if (!job.active || job.K > (unsigned long long)GNC_SERIAL_MAX) return;
  if (job.point_flags)
    for (int i = threadIdx.x; i < job.n_points; i += 128) job.point_flags[i] = 0;
  __syncthreads();
  if (threadIdx.x == 0) gnc_tls_serial(job);
}

// Sum (slot RED_MAX: max) of 16 values per thread over the CTA and the cluster, in a fixed order.  Warp level: a
// transposed butterfly -- every exchange halves the values a lane carries, 16 shuffles instead of 16 x 5 -- after
// which lane 2 i holds the warp's result i; CTA level: warp 0 adds the warps' results as a fixed tree, lane i
// ending with result i; cluster level: the same lanes add the peers' results in rank order through distributed
// shared memory.  On return sm->total is valid FOR WARP 0 ONLY (the caller's next barrier publishes it).
// NC == 0 ("grid mode", few registrations with very many line vectors): gridDim.x CTAs per registration, launched
// cooperatively (all resident); the CTAs' results meet in a global scratch behind a counter barrier, every CTA adding
// them up in rank order.
struct GridRed {
  double* red;        // [2][gridDim.x][GNC_NRED], double-buffered by reduction parity
  unsigned int* bar;  // arrivals so far (zeroed by gnc_tls_small_kernel, which runs before on the same stream)
};
template <int NC, int T>
__device__ __forceinline__ void block_reduce16(GncSmem* sm, double (&v)[GNC_NRED], int& red_no, const GridRed& gr) {
  const int parity = red_no & 1;
  constexpr int NW = T / 32, NH = NW / 2;
  static_assert(NW >= 2 && NW <= GNC_MAX_WARPS && (NW & (NW - 1)) == 0, "");
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  bool top = true;  // this lane carries slot RED_MAX in its last value
#define PSU_RSTEP(OFF, N)                                             \
  {                                                                   \
    const bool up = (lane & OFF) != 0;                                \
    top = top && up;                                                  \
    _Pragma("unroll") for (int i = 0; i < N; ++i) {                   \
      const double send = up ? v[i] : v[i + N];                       \
      const double keep = up ? v[i + N] : v[i];                       \
      const double recv = __shfl_xor_sync(0xffffffffu, send, OFF);    \
      v[i] = (i == N - 1 && top) ? fmax(keep, recv) : keep + recv;    \
    }                                                                 \
  }
  PSU_RSTEP(16, 8)
  PSU_RSTEP(8, 4)
  PSU_RSTEP(4, 2)
  PSU_RSTEP(2, 1)
#undef PSU_RSTEP
  {
    const double o = __shfl_xor_sync(0xffffffffu, v[0], 1);
    v[0] = top ? fmax(v[0], o) : v[0] + o;
  }
  if ((lane & 1) == 0) sm->warp_part[wid][lane >> 1] = v[0];
  __syncthreads();
  if (wid == 0) {
    const int idx = lane & 15, half = lane >> 4;
    const bool is_max = idx == RED_MAX;
    double a[NH];
#pragma unroll
    for (int j = 0; j < NH; ++j) a[j] = sm->warp_part[half * NH + j][idx];
#pragma unroll
    for (int s = 1; s < NH; s <<= 1)
#pragma unroll
      for (int j = 0; j + s < NH; j += 2 * s) a[j] = is_max ? fmax(a[j], a[j + s]) : a[j] + a[j + s];
    const double y = __shfl_xor_sync(0xffffffffu, a[0], 16);
    const double lo = half ? y : a[0], hi = half ? a[0] : y;
    const double x = is_max ? fmax(lo, hi) : lo + hi;
    if (lane < 16) {
      sm->part[parity][idx] = x;
      if (NC == 1) sm->total[idx] = x;
    }
    if (NC == 0) {
      const unsigned G = gridDim.x;
      double* __restrict__ buf = gr.red + (size_t)parity * G * GNC_NRED;
      if (lane < 16) __stcg(buf + (size_t)blockIdx.x * GNC_NRED + lane, x);
      __threadfence();  // the partial results before the arrival
      __syncwarp();
      if (lane == 0) {
        atomicAdd(gr.bar, 1u);
        const unsigned target = ((unsigned)red_no + 1u) * G;
        unsigned seen;
        do {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(gr.bar) : "memory");
          if (seen < target) __nanosleep(64);
        } while (seen < target);
      }
      __syncwarp();
      {
        // lane = result + 16 x half: each half adds its share of the ranks in order, eight loads in flight at a time
        // (the additions wait for the loads: one load at a time would cost an L2 round trip per CTA of the registration)
        const unsigned half_n = (G + 1) / 2, r_lo = half * half_n, r_hi = (r_lo + half_n < G) ? r_lo + half_n : G;
        double acc = is_max ? -INFINITY : 0.0;
        for (unsigned r = r_lo; r < r_hi; r += 8) {
          double y[8];
#pragma unroll
          for (unsigned j = 0; j < 8; ++j) y[j] = (r + j < r_hi) ? __ldcg(buf + (size_t)(r + j) * GNC_NRED + idx) : (is_max ? -INFINITY : 0.0);
#pragma unroll
          for (unsigned j = 0; j < 8; ++j) acc = is_max ? fmax(acc, y[j]) : acc + y[j];
        }
        const double other = __shfl_xor_sync(0xffffffffu, acc, 16);
        const double a_lo = half ? other : acc, a_hi = half ? acc : other;
        if (lane < 16) sm->total[idx] = is_max ? fmax(a_lo, a_hi) : a_lo + a_hi;
      }
    }
  }
  if (NC > 1) {
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();
    if (wid == 0 && lane < 16) {
      double acc = 0.0;
#pragma unroll
      for (int r = 0; r < NC; ++r) {
        const GncSmem* peer = cluster.map_shared_rank(sm, r);
        const double x = peer->part[parity][lane];
        acc = (r == 0) ? x : ((lane == RED_MAX) ? fmax(acc, x) : acc + x);
      }
      sm->total[lane] = acc;
    }
  }
  if (wid == 0) __syncwarp();
  ++red_no;
}

template <int NC, int T, int CPS>
__global__ void __launch_bounds__(T, CPS)
    gnc_tls_kernel(const GncJob* __restrict__ jobs, int cap_per_cta, const double GNC_DEEP_MARGIN) {
  constexpr int NW = T / 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GncSmem* sm = reinterpret_cast<GncSmem*>(smem_raw);
  double* lvs = reinterpret_cast<double*>(smem_raw + ((sizeof(GncSmem) + 15) & ~size_t(15)));
  const GncJob& job = jobs[blockIdx.y];
  if (!job.active) return;  // uniform over the cluster
  if (job.K <= (unsigned long long)GNC_SERIAL_MAX) return;  // gnc_tls_small_kernel's (uniform over the cluster)
  const long long t_kernel0 = clock64();
  const int max_iterations = job.max_iterations;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const unsigned rank = (NC > 1) ? cg::this_cluster().block_rank() : (NC == 0 ? blockIdx.x : 0u);
  const unsigned NCTA = (NC == 0) ? gridDim.x : (unsigned)NC;  // CTAs of this registration
  const GridRed gr = {job.grid_red, job.grid_bar};
  const unsigned long long K = job.K;
  // contiguous slice of the line vectors for this CTA, cut into one contiguous segment per warp
  const unsigned long long per = ((K + NCTA - 1) / NCTA + 63) & ~63ull;
  const unsigned long long k_lo = (per * rank < K) ? per * rank : K;
  const unsigned long long k_hi = (k_lo + per < K) ? k_lo + per : K;
  const int nloc = (int)(k_hi - k_lo);
  // The slice is dealt to the warps in blocks of 64 line vectors, round robin: position l of warp w is the slice's
  // line vector PH(l) = ((l / 64) NW + w) 64 + l % 64, so that the warps of a CTA, walking their positions in step,
  // stream one contiguous run of NW x 64 line vectors per array (whole DRAM rows), not NW scattered ones.
#define PH(l) ((((l) >> 6) * NW + wid) * 64 + ((l) & 63))
  // positions of this warp among the slice's first m line vectors
  auto owned = [&](int m) -> int {
    const int nb = m >> 6, rem = m & 63;
    return (nb / NW + (wid < nb % NW ? 1 : 0)) * 64 + ((nb % NW) == wid ? rem : 0);
  };
  const int n_w0 = owned(nloc);
  // positions [0, cs) of a warp live in shared memory: comps 0..5 and the slot, [7][cs]
  const int cs = (cap_per_cta / NW) & ~63;  // (whole steps)
  double* __restrict__ wsm = lvs + (size_t)wid * 7 * cs;
  double* __restrict__ lvg = job.lv;
  const unsigned long long lv_cap = lvg ? job.lv_cap : 0ull;
  const size_t st = (size_t)lv_cap;
  double* __restrict__ g0 = lvg ? lvg + k_lo : nullptr;  // component c of position l: g0[c * st + PH(l)]
  double* __restrict__ gwl = job.weights + k_lo;         // slots of the positions that are not in shared memory
  uint32_t* __restrict__ gpl = job.perm ? job.perm + k_lo : nullptr;  // original (slice-local) index of a position
  // positions [cs, gh) have a home in the global scratch; what lies beyond is re-formed from the points every pass
  const int gh0 = (lvg && lv_cap > k_lo) ? owned((lv_cap - k_lo < (unsigned long long)nloc) ? (int)(lv_cap - k_lo) : nloc) : 0;
  const bool can_compact = lvg != nullptr && gpl != nullptr && k_hi <= lv_cap;

  double nb2 = job.noise_bound * job.noise_bound;
  if (nb2 < 1e-16) nb2 = 1e-2;  // registration.cc:1592-1595

  // (the operands of the cold paths stay in the job record: registers are what the streaming loop is short of)
  auto form = [&](int p, double sv[3], double tv[3]) {  // p: slice-local index
    const uint2 e = job.edges[k_lo + p];
    if (job.pts8)
      load_lv8(job.pts8, e, job.inv_scale, sv, tv);
    else
      load_lv(job.src, job.dst, e, job.inv_scale, sv, tv);
  };

  int red_no = 0;  // reductions so far (their parity double-buffers the partial results peers read)
  int n_w = n_w0, it_done = 0;
  bool permuted = false, unit = true;
  if (tid == 0) {
    sm->t_stream = sm->t_svd = sm->sum_act = sm->t_prologue = sm->t_start = 0;
    sm->n_armed = 0;
    sm->first_armed = -1;
  }
  int n_reopened = 0;
  {
    const bool sleeping = can_compact && job.gnc_factor > 1.0;  // th1 must not grow
    const bool ready = job.lv_ready && lvg != nullptr;
    const int gh = gh0;
    double acc[GNC_NRED];
#pragma unroll
    for (int i = 0; i < GNC_NRED; ++i) acc[i] = 0.0;
    acc[RED_MAX] = -INFINITY;
    // ---- prologue: every position into its home, H_0 = sum sv tv^T (unit weights)
    for (int base = 0; base < n_w; base += 64) {
      const int la = base + lane, lb = la + 32;
      const bool va = la < n_w, vb = lb < n_w;
      double sa[3], ta[3], sb[3], tb[3];
      auto get = [&](int l, double sv[3], double tv[3]) {
        const int p = PH(l);
        if (ready && l < gh) {
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            sv[r] = __ldcg(g0 + r * st + p);
            tv[r] = __ldcg(g0 + (3 + r) * st + p);
          }
        } else {
          form(p, sv, tv);
        }
      };
      auto put = [&](int l, const double sv[3], const double tv[3]) {
        if (l < cs) {
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            wsm[r * cs + l] = sv[r];
            wsm[(3 + r) * cs + l] = tv[r];
          }
        } else if (l < gh && !ready) {
          const int p = PH(l);
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            __stcg(g0 + r * st + p, sv[r]);
            __stcg(g0 + (3 + r) * st + p, tv[r]);
          }
        }
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int c = 0; c < 3; ++c) acc[r * 3 + c] = fma(sv[r], tv[c], acc[r * 3 + c]);
      };
      if (ready && (lane & 3) == 0) {
        const int pa = la + 64 * GNC_PF_STEPS, pb = lb + 64 * GNC_PF_STEPS;
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          if (pa < gh) asm volatile("prefetch.global.L2 [%0];" ::"l"(g0 + r * st + PH(pa)));
          if (pb < gh) asm volatile("prefetch.global.L2 [%0];" ::"l"(g0 + r * st + PH(pb)));
        }
      }
      if (va) get(la, sa, ta);
      if (vb) get(lb, sb, tb);
      if (va) put(la, sa, ta);
      if (vb) put(lb, sb, tb);
    }
    if (tid < 9) sm->Vw[tid] = (tid % 4 == 0) ? 1.0 : 0.0;
    if (tid == 0) {
      sm->drift = 0.0;
      sm->min_wake = INFINITY;
      sm->mu = 1.0;
      sm->prev_cost = INFINITY;
      sm->cost = INFINITY;
    }
    if (job.use_init) {
      if (tid < 9) sm->R[tid] = job.R_init[(tid % 3) * 3 + tid / 3];  // column-major -> row-major
    } else {
      block_reduce16<NC, T>(sm, acc, red_no, gr);
      if (tid == 0) svd_from_smem(sm);
    }
    __syncthreads();
    if (tid == 0) {
      sm->t_prologue = clock64() - t_kernel0;
      sm->t_start = clock64();
    }

    // position l of this warp's segment: line vector, previous slot, original index
    auto fetch = [&](int l, bool armed, double sv[3], double tv[3], double& slot, uint32_t& idx) {
      if (l < cs) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          sv[r] = wsm[r * cs + l];
          tv[r] = wsm[(3 + r) * cs + l];
        }
        if (!unit) slot = wsm[6 * cs + l];
      } else if (l < gh) {
        const int p = PH(l);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          sv[r] = __ldcg(g0 + r * st + p);
          tv[r] = __ldcg(g0 + (3 + r) * st + p);
        }
        if (!unit) slot = __ldcg(gwl + p);
      } else {
        const int p = PH(l);
        form(p, sv, tv);
        if (!unit) slot = __ldcg(gwl + p);
      }
      if (armed) idx = permuted ? __ldcg(gpl + PH(l)) : (uint32_t)PH(l);
    };
    auto put_slot = [&](int l, double v) {
      if (l < cs)
        wsm[6 * cs + l] = v;
      else
        __stcg(gwl + PH(l), v);
    };
    // line vector, slot and original index into position r (parking, reopening)
    auto put_all = [&](int r, const double sv[3], const double tv[3], double slot, uint32_t idx) {
      const int p = PH(r);
      if (r < cs) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          wsm[c * cs + r] = sv[c];
          wsm[(3 + c) * cs + r] = tv[c];
        }
        wsm[6 * cs + r] = slot;
      } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          __stcg(g0 + c * st + p, sv[c]);
          __stcg(g0 + (3 + c) * st + p, tv[c]);
        }
        __stcg(gwl + p, slot);
      }
      __stcg(gpl + p, idx);
    };

    for (int it = 0; it < max_iterations; ++it) {
      it_done = it + 1;
      // (the rotation and the pass constants are read from shared memory where they are used: broadcast loads
      // are cheap, the 30 registers they would occupy across the pass are not)
      const double* __restrict__ R = sm->R;
      if (it == 0) {
        // mu initialisation needs max r^2 first (registration.cc:1628-1639)
        double mx = 0.0;
        for (int base = 0; base < n_w; base += 64) {
          const int la = base + lane, lb = la + 32;
          double sa[3], ta[3], sb[3], tb[3], w_ = 0.0;
          uint32_t i_ = 0;
          if ((lane & 3) == 0) {
            const int pa = la + 64 * GNC_PF_STEPS, pb = lb + 64 * GNC_PF_STEPS;
#pragma unroll
            for (int r = 0; r < 6; ++r) {
              if (pa >= cs && pa < gh) asm volatile("prefetch.global.L2 [%0];" ::"l"(g0 + r * st + PH(pa)));
              if (pb >= cs && pb < gh) asm volatile("prefetch.global.L2 [%0];" ::"l"(g0 + r * st + PH(pb)));
            }
          }
          if (la < n_w) fetch(la, false, sa, ta, w_, i_);
          if (lb < n_w) fetch(lb, false, sb, tb, w_, i_);
          if (la < n_w) mx = fmax(mx, residual2(R, sa, ta));
          if (lb < n_w) mx = fmax(mx, residual2(R, sb, tb));
        }
#pragma unroll
        for (int i = 0; i < GNC_NRED; ++i) acc[i] = 0.0;
        acc[RED_MAX] = mx;
        block_reduce16<NC, T>(sm, acc, red_no, gr);
        if (tid == 0) {
          const double max_residual = sm->total[RED_MAX];
          const double mu = 1.0 / (2.0 * max_residual / nb2 - 1.0);
          sm->mu = mu;
          GncCtl c;
          c.th1 = (mu + 1.0) / mu * nb2;
          c.th2 = mu / (mu + 1.0) * nb2;
          c.sqrt_wnum = sqrt(nb2 * mu * (mu + 1.0));
          c.mu = mu;
          c.drift = 0.0;
          c.sqrt_th1_up = sqrtf((float)c.th1) * 1.000001f;
          c.stop = (mu <= 0.0) ? 2 : 0;  // degenerate: residuals already tiny; weights stay 1, R stays
          c.armed = 0;
          c.reopen = 0;
          sm->ctl = c;
        }
        __syncthreads();
        if (sm->ctl.stop) break;
      }
      const GncCtl& ctl = sm->ctl;
      const bool armed = ctl.armed != 0;
#pragma unroll
      for (int i = 0; i < GNC_NRED; ++i) acc[i] = 0.0;
      acc[RED_MAX] = -INFINITY;
      int n_deep = 0;  // deep sleepers this lane left in the range
      // one line vector: cost term with the previous weight, closed-form new weight, H += w sv tv^T.
      // slot >= 0: the previous weight; slot < 0: weight 0, asleep until the drift reaches -slot.  A deep sleeper
      // (remaining margin >= GNC_DEEP_MARGIN) is skipped: its weight was 0 and provably still is.
      auto eval = [&](const double sv[3], const double tv[3], double slot, bool& deep) -> double {
        const double drift = ctl.drift;
        if (slot < 0.0 && (-slot - drift) >= GNC_DEEP_MARGIN) {
          deep = true;
          return slot;
        }
        deep = false;
        const double r2 = residual2(R, sv, tv);
        acc[RED_COST] = fma(fmax(slot, 0.0), r2, acc[RED_COST]);  // cost uses the previous weights (registration.cc:1648)
        // sqrt(eps^2 mu (mu + 1) / r^2) - mu  (registration.cc:1655), selected between the two plateaus; H takes the
        // term unconditionally (w = 0 adds exact zeros): one branch per line vector instead of four
        double wn = fma(ctl.sqrt_wnum, rsqrt_pos(r2), -ctl.mu);
        wn = (r2 <= ctl.th2) ? 1.0 : wn;
        wn = (r2 >= ctl.th1) ? 0.0 : wn;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const double xs = sv[r] * wn;
#pragma unroll
          for (int c = 0; c < 3; ++c) acc[r * 3 + c] = fma(xs, tv[c], acc[r * 3 + c]);
        }
        if (wn != 0.0 || !sleeping) return wn;
        // the margin in units of rotation change.  A LOWER bound is all that is needed, so it is formed in FP32
        // (two MUFU operations) and shaved by far more than the FP32 rounding of r, sqrt(th1) and |sv|.
        const float s2f = (float)fma(sv[2], sv[2], fma(sv[1], sv[1], sv[0] * sv[0]));
        const float mf = (sqrtf((float)r2) - ctl.sqrt_th1_up) * rsqrtf(s2f) * 0.999f - 1e-6f;
        const double out = (mf > 0.0f && mf < 1e30f) ? -(drift + (double)mf) : 0.0;
        deep = out < 0.0 && (-out - drift) >= GNC_DEEP_MARGIN;
        return out;
      };
      const long long c_stream0 = (tid == 0) ? clock64() : 0ll;
      int cnt = 0;  // armed pass: positions kept so far (warp-uniform)
      // One step = 64 positions of the warp (two coalesced groups in flight per lane).  TIER 0: the step lies in
      // shared memory, TIER 1: in the global scratch -- both complete, no per-lane tests; TIER 2: anything else (the
      // last, partial step; positions without a home).  ARMED steps also park (see the header comment).
      auto step = [&](auto TIER_, auto ARMED_, const int base) {
        constexpr int TIER = decltype(TIER_)::value;
        constexpr bool ARMED = decltype(ARMED_)::value;
        const int la = base + lane, lb = la + 32;
        const bool va = TIER < 2 || la < n_w, vb = TIER < 2 || lb < n_w;
        double sa[3], ta[3], sb[3], tb[3], wa = 1.0, wb = 1.0;
        uint32_t ia = 0, ib = 0;
        const int p0 = ((base >> 6) * NW + wid) * 64 + lane;  // = PH(la); PH(lb) = p0 + 32
        if (TIER == 0) {
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            sa[r] = wsm[r * cs + la];
            ta[r] = wsm[(3 + r) * cs + la];
            sb[r] = wsm[r * cs + lb];
            tb[r] = wsm[(3 + r) * cs + lb];
          }
          if (!unit) {
            wa = wsm[6 * cs + la];
            wb = wsm[6 * cs + lb];
          }
          if (ARMED) {
            ia = permuted ? __ldcg(gpl + p0) : (uint32_t)p0;
            ib = permuted ? __ldcg(gpl + p0 + 32) : (uint32_t)(p0 + 32);
          }
        } else if (TIER == 1) {
          const double* __restrict__ ga = g0 + p0;
          // register-free look-ahead: the sectors this warp reads in a later step are pulled into L2 (one lane per
          // 32-byte sector issues the prefetch), so that the loads below see L2 latency instead of HBM's
          if ((lane & 3) == 0 && base + 64 * GNC_PF_STEPS + 64 <= n_w) {
            const double* __restrict__ gp = ga + (size_t)(GNC_PF_STEPS * NW * 64);
#pragma unroll
            for (int r = 0; r < 6; ++r) {
              asm volatile("prefetch.global.L2 [%0];" ::"l"(gp + r * st));
              asm volatile("prefetch.global.L2 [%0];" ::"l"(gp + r * st + 32));
            }
            if (!unit) {
              asm volatile("prefetch.global.L2 [%0];" ::"l"(gwl + p0 + GNC_PF_STEPS * NW * 64));
              asm volatile("prefetch.global.L2 [%0];" ::"l"(gwl + p0 + GNC_PF_STEPS * NW * 64 + 32));
            }
          }
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            sa[r] = __ldcg(ga + r * st);
            ta[r] = __ldcg(ga + (3 + r) * st);
            sb[r] = __ldcg(ga + r * st + 32);
            tb[r] = __ldcg(ga + (3 + r) * st + 32);
          }
          if (!unit) {
            wa = __ldcg(gwl + p0);
            wb = __ldcg(gwl + p0 + 32);
          }
          if (ARMED) {
            ia = permuted ? __ldcg(gpl + p0) : (uint32_t)p0;
            ib = permuted ? __ldcg(gpl + p0 + 32) : (uint32_t)(p0 + 32);
          }
        } else {
          if (va) fetch(la, ARMED, sa, ta, wa, ia);
          if (vb) fetch(lb, ARMED, sb, tb, wb, ib);
        }
        bool da = false, db = false;
        double oa = 0.0, ob = 0.0;
        if (va) oa = eval(sa, ta, wa, da);
        if (vb) ob = eval(sb, tb, wb, db);
        if (!ARMED) {
          n_deep += (da ? 1 : 0) + (db ? 1 : 0);
          if (TIER == 0) {
            wsm[6 * cs + la] = oa;
            wsm[6 * cs + lb] = ob;
          } else if (TIER == 1) {
            __stcg(gwl + p0, oa);
            __stcg(gwl + p0 + 32, ob);
          } else {
            if (va) put_slot(la, oa);
            if (vb) put_slot(lb, ob);
          }
        } else {
          // the deep sleepers leave the range: the others move down inside the warp's own positions, in order (every
          // store lands at or below the positions this step loaded, all of them loaded before the votes)
          const bool ka = va && !da, kb = vb && !db;
          const unsigned ma = __ballot_sync(0xffffffffu, ka), mb = __ballot_sync(0xffffffffu, kb);
          __syncwarp();
          if (va && da) acc[RED_MAX] = fmax(acc[RED_MAX], oa);  // max of the negated wake-up drifts = -(the smallest)
          if (vb && db) acc[RED_MAX] = fmax(acc[RED_MAX], ob);
          if (ka) put_all(cnt + __popc(ma & lt_mask), sa, ta, oa, ia);
          cnt += __popc(ma);
          if (kb) put_all(cnt + __popc(mb & lt_mask), sb, tb, ob, ib);
          cnt += __popc(mb);
        }
      };
      auto sweep = [&](auto ARMED_) {
        using I0 = std::integral_constant<int, 0>;
        using I1 = std::integral_constant<int, 1>;
        using I2 = std::integral_constant<int, 2>;
        const int nS = (cs < n_w ? cs : n_w) & ~63;
        int base = 0;
        for (; base < nS; base += 64) step(I0{}, ARMED_, base);
        if (base == cs) {
          const int nG = (gh < n_w ? gh : n_w) & ~63;
          for (; base < nG; base += 64) step(I1{}, ARMED_, base);
        }
        for (; base < n_w; base += 64) step(I2{}, ARMED_, base);
      };
      if (armed)
        sweep(std::true_type{});
      else
        sweep(std::false_type{});
      if (tid == 0) {
        sm->t_stream += clock64() - c_stream0;
        sm->sum_act += n_w;
        if (armed) {
          ++sm->n_armed;
          if (sm->first_armed < 0) sm->first_armed = it;
        }
      }
      if (armed) {
        n_w = cnt;
        permuted = true;
      }
      unit = false;
      acc[RED_LEFT] = (lane == 0) ? (double)n_w : 0.0;  // positions left in the warp's range
      acc[RED_DEEP] = (double)n_deep;
      block_reduce16<NC, T>(sm, acc, red_no, gr);
      if (tid == 0) {
        const double cost = sm->total[RED_COST];
        const double cost_diff = fabs(cost - sm->prev_cost);
        const double mu_n = sm->mu * job.gnc_factor;
        sm->mu = mu_n;
        sm->prev_cost = cost;
        sm->cost = cost;
        GncCtl c;
        c.stop = (cost_diff < job.cost_threshold || it + 1 >= max_iterations) ? 1 : 0;
        c.armed = 0;
        c.reopen = 0;
        c.th1 = c.th2 = c.sqrt_wnum = 0.0;
        c.mu = mu_n;
        c.drift = sm->drift;
        c.sqrt_th1_up = 0.f;
        if (!c.stop) {
          const long long c0 = clock64();
          rotation_from_smem(sm);
          sm->t_svd += clock64() - c0;
          sm->min_wake = fmin(sm->min_wake, -sm->total[RED_MAX]);
          if (sm->min_wake <= sm->drift) {  // (uniform over the cluster: same drift, cluster-wide minimum)
            c.reopen = 1;
            sm->min_wake = INFINITY;
          }
          c.th1 = (mu_n + 1.0) / mu_n * nb2;
          c.th2 = mu_n / (mu_n + 1.0) * nb2;
          c.sqrt_wnum = sqrt(nb2 * mu_n * (mu_n + 1.0));
          c.drift = sm->drift;
          c.sqrt_th1_up = sqrtf((float)c.th1) * 1.000001f;
          // park when enough of this CTA's positions sleep deeply (its own counts, before the cluster combined them)
          const double deep = sm->part[(red_no - 1) & 1][RED_DEEP], left = sm->part[(red_no - 1) & 1][RED_LEFT];
          c.armed = (sleeping && !c.reopen && left >= 256.0 && deep * 100.0 >= left * (double)GNC_PARK_PCT) ? 1 : 0;
        }
        sm->ctl = c;
      }
      __syncthreads();
      if (sm->ctl.stop) break;
      if (sm->ctl.reopen && permuted) {
        // Rare (the rotation jumped by more than the parking margin after line vectors were parked): every parked
        // line vector returns to its warp's range, re-formed from its endpoints, with slot 0 ("weight 0, awake" --
        // exactly its state).  The positions left are marked by original index; what is not marked was parked.
        ++n_reopened;
        unsigned char* __restrict__ mark = reinterpret_cast<unsigned char*>(job.perm + lv_cap) + k_lo;
        for (int l = tid; l < nloc; l += T) __stcg(mark + l, (unsigned char)0);
        __syncthreads();
        for (int l = lane; l < n_w; l += 32) __stcg(mark + __ldcg(gpl + PH(l)), (unsigned char)1);
        __syncthreads();
        int cnt = n_w;
        for (int base = 0; base < n_w0; base += 32) {
          const int q = base + lane;
          const int p = PH(q);
          const bool missing = q < n_w0 && __ldcg(mark + p) == 0;
          const unsigned m = __ballot_sync(0xffffffffu, missing);
          if (missing) {
            double sv[3], tv[3];
            form(p, sv, tv);
            put_all(cnt + __popc(m & lt_mask), sv, tv, 0.0, (uint32_t)p);
          }
          cnt += __popc(m);
        }
        n_w = cnt;
        __syncthreads();
      }
    }
  }

  const long long t_loop_end = (tid == 0) ? clock64() : 0ll;
  // ---- epilogue: inlier mask w >= 0.5 (all when <= 10), endpoint flags (registration.cc:1676-1691,
  // :1114-1155).  The stale-bit defect of the reference is resolved as "zero then set".  Parked line vectors sit
  // at weight 0; the positions left carry their original index.
  {
    double cntv[GNC_NRED];
#pragma unroll
    for (int i = 0; i < GNC_NRED; ++i) cntv[i] = 0.0;
    auto slot_at = [&](int l) -> double { return unit ? 1.0 : ((l < cs) ? wsm[6 * cs + l] : __ldcg(gwl + PH(l))); };
    for (int l = lane; l < n_w; l += 32) cntv[0] += (slot_at(l) >= 0.5) ? 1.0 : 0.0;  // < 0: asleep, weight 0
    if (job.point_flags) {
      // zero this cluster's share of the flags before anyone sets them (the reduction synchronises the cluster)
      for (int i = rank * T + tid; i < job.n_points; i += NCTA * T) job.point_flags[i] = 0;
    }
    block_reduce16<NC, T>(sm, cntv, red_no, gr);
    __syncthreads();
    const long long gf = (long long)(sm->total[0] + 0.5);
    const bool all_in = gf <= 10;
    if (all_in || permuted) {
      // every line vector of the slice at once: inlier (all_in) or not (the parked ones; the rest is set below)
      for (int l = tid; l < nloc; l += T) {
        if (job.inliers) job.inliers[k_lo + l] = all_in ? 1 : 0;
        if (all_in && job.point_flags) {
          const uint2 e = job.edges[k_lo + l];
          job.point_flags[e.x] = 1;
          job.point_flags[e.y] = 1;
        }
      }
      __syncthreads();
    }
    if (!all_in) {
      for (int l = lane; l < n_w; l += 32) {
        const bool in = slot_at(l) >= 0.5;
        const size_t k = (size_t)k_lo + (permuted ? (size_t)__ldcg(gpl + PH(l)) : (size_t)PH(l));  // original index
        if (job.inliers && (in || !permuted)) job.inliers[k] = in ? 1 : 0;
        if (in && job.point_flags) {
          const uint2 e = job.edges[k];
          job.point_flags[e.x] = 1;
          job.point_flags[e.y] = 1;
        }
      }
    }
    if (rank == 0 && tid == 0) {
      if (job.R_out) {
        for (int c = 0; c < 3; ++c)
          for (int r = 0; r < 3; ++r) job.R_out[c * 3 + r] = sm->R[r * 3 + c];  // column-major out
      }
      if (job.info) {
        job.info[0] = it_done;
        job.info[1] = (int)(all_in ? (long long)K : gf);
        job.info[2] = n_reopened;                          // times the parked line vectors had to return
        job.info[3] = (int)((clock64() - sm->t_start) >> 4);  // GNC loop cycles / 16 (diagnostic)
      }
      if (job.cost) job.cost[0] = sm->cost;
      if (job.prof) {
        job.prof[0] = sm->t_stream;
        job.prof[1] = t_loop_end - sm->t_start;
        job.prof[2] = sm->t_svd;
        job.prof[3] = (long long)cs * NW;
        job.prof[4] = sm->t_prologue;           // prologue: line vectors into their homes, H_0, first SVD
        job.prof[5] = clock64() - t_loop_end;  // epilogue: inlier mask, endpoint flags
        job.prof[6] = sm->sum_act * NW;         // positions of warp 0 summed over the passes, times the warps
        job.prof[7] = sm->n_armed + 100 * (sm->first_armed + 1) + 10000 * (long long)n_reopened;
      }
    }
  }
#undef PH
  if (NC > 1) cg::this_cluster().sync();  // peers may still be reading this CTA's partial sums
}

// ------------------------------------------------------------------------------------------
// batched closed-form Kabsch: one warp per hypothesis
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    kabsch_batch_kernel(const double* __restrict__ src, const double* __restrict__ dst, const uint2* __restrict__ edges,
                        const uint32_t* __restrict__ sets, int k, unsigned long long n_hyp, double* __restrict__ Rout,
                        double* __restrict__ tout) {
  const unsigned long long h = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (h >= n_hyp) return;
  double H[9], cs[3] = {0, 0, 0}, cd[3] = {0, 0, 0};
#pragma unroll
  for (int i = 0; i < 9; ++i) H[i] = 0.0;
  for (int l = lane; l < k; l += 32) {
    const uint2 e = edges[sets[h * (unsigned long long)k + l]];
    double sv[3], tv[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const double sa = src[3 * (size_t)e.x + r], sb = src[3 * (size_t)e.y + r];
      const double da = dst[3 * (size_t)e.x + r], db = dst[3 * (size_t)e.y + r];
      sv[r] = sb - sa;
      tv[r] = db - da;
      cs[r] += sa + sb;
      cd[r] += da + db;
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) H[r * 3 + c] += sv[r] * tv[c];
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) H[i] = warp_sum(H[i]);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    cs[r] = warp_sum(cs[r]);
    cd[r] = warp_sum(cd[r]);
  }
  if (lane == 0) {
    double Hm[3][3], R[3][3];
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) Hm[r][c] = H[r * 3 + c];
    kabsch_rotation(Hm, R);
    for (int c = 0; c < 3; ++c)
      for (int r = 0; r < 3; ++r) Rout[h * 9 + c * 3 + r] = R[r][c];
    if (tout) {
      const double invn = 1.0 / (2.0 * (double)k);
      for (int r = 0; r < 3; ++r)
        tout[h * 3 + r] = cd[r] * invn - ((R[r][0] * cs[0] + R[r][1] * cs[1]) + R[r][2] * cs[2]) * invn;
    }
  }
}

int gnc_capacity_for(int ctas_per_sm, int warps);
size_t gnc_smem_bytes(int cap) { return ((sizeof(GncSmem) + 15) & ~size_t(15)) + (size_t)7 * cap * sizeof(double); }

template <int NC, int T, int CPS>
int launch_gnc_nc(cudaStream_t st, const GncJob* d_jobs, int n_jobs, int cap_per_cta, int grid_ctas = 0) {
  static bool attr_set = false;
  const int max_cap = gnc_capacity_for(CPS, T / 32);
  if (cap_per_cta > max_cap) cap_per_cta = max_cap;
  const size_t smem = gnc_smem_bytes(cap_per_cta);
  if (!attr_set) {
    PSU_CUDA(cudaFuncSetAttribute(gnc_tls_kernel<NC, T, CPS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)gnc_smem_bytes(gnc_capacity_for(CPS, T / 32))));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(NC > 0 ? NC : (unsigned)grid_ctas, (unsigned)n_jobs, 1);
  cfg.blockDim = dim3(T, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  if (NC > 0) {
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = NC;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
  } else {
    attr[0].id = cudaLaunchAttributeCooperative;  // all CTAs resident: they wait for one another
    attr[0].val.cooperative = 1;
  }
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // (a performance knob only -- any value gives the same results; the tests shrink the margin to force wake-ups)
  const double deep_margin = debug_knobs().gnc_deep_margin > 0.0 ? debug_knobs().gnc_deep_margin : GNC_DEEP_MARGIN_DEFAULT;
  PSU_CUDA(cudaLaunchKernelEx(&cfg, gnc_tls_kernel<NC, T, CPS>, d_jobs, cap_per_cta, deep_margin));
  return PSULVSB_OK;
}

}  // namespace

namespace {
int gnc_capacity_for(int ctas_per_sm, int warps) {
  // the CTAs resident on an SM share its 227 KB (232 448 bytes; 1 KB per resident CTA is the system's); every warp
  // caches whole steps of 64 positions: 16 warps x 256 positions x 56 bytes fit one 512-thread CTA per SM exactly
  const size_t budget = (size_t)232448 / (size_t)ctas_per_sm - (ctas_per_sm > 1 ? 1024 : 0);
  const size_t fixed = (sizeof(GncSmem) + 15) & ~size_t(15);
  int cap = (int)((budget - fixed) / (7 * sizeof(double)));
  cap -= cap % (64 * warps);  // (whole steps of 64 positions per warp)
  return cap;
}
}  // namespace

int gnc_default_capacity() { return gnc_capacity_for(1, 16); }

// CTAs per hypothesis for a batch of n_jobs: as many SMs per job as keeps the whole batch resident
int gnc_cluster_for(int n_jobs) {
  const int slots = sm_count() * GNC_CTAS_PER_SM;
  if (n_jobs * 8 <= slots) return 8;
  if (n_jobs * 4 <= slots) return 4;
  if (n_jobs * 2 <= slots) return 2;
  return 1;
}

int launch_gnc_tls(cudaStream_t st, const GncJob* d_jobs, int n_jobs, int cap_per_cta, int cluster, int n_active) {
  if (n_jobs <= 0) return PSULVSB_OK;
  if (n_active <= 0 || n_active > n_jobs) n_active = n_jobs;  // jobs that are not marked inactive (their CTAs exit at once)
  gnc_tls_small_kernel<<<n_jobs, 128, 0, st>>>(d_jobs);  // tiny subsets: the reference's arithmetic replayed by one thread
  PSU_CHECK_LAUNCH("gnc_tls_small_kernel");
  if (cap_per_cta < 32) cap_per_cta = 32;
  if (cluster > 8) {  // grid mode: `cluster` CTAs per registration (the jobs must carry grid_red / grid_bar)
    if ((long long)cluster * n_jobs > (long long)sm_count())
      return fail(PSULVSB_ERR_INVALID, "launch_gnc_tls: grid mode needs CTAs per registration x registrations <= SMs");
    return launch_gnc_nc<0, 512, 1>(st, d_jobs, n_jobs, cap_per_cta, cluster);
  }
  switch (cluster) {
    // (measured: 512 threads x 2 CTAs per SM = 64 registers spills 1.3 KB per thread and loses 25 %)
    case 8:
      // few registrations (8 CTAs each still leave SMs idle): 512 threads, one CTA per SM -- half the line
      // vectors per thread in the latency-bound pass
      if (n_jobs * 8 <= sm_count()) return launch_gnc_nc<8, 512, 1>(st, d_jobs, n_jobs, cap_per_cta);
      return launch_gnc_nc<8, 256, 2>(st, d_jobs, n_jobs, cap_per_cta);
    case 4: return launch_gnc_nc<4, 256, 2>(st, d_jobs, n_jobs, cap_per_cta);
    case 2: return launch_gnc_nc<2, 256, 2>(st, d_jobs, n_jobs, cap_per_cta);
    case 1: {
      // one CTA per hypothesis (large batches): 512 threads per SM in all, cut into as many CTAs as it takes to have the
      // whole launch resident at once (up to four 128-thread CTAs per SM) -- one registration's serial phases (reductions,
      // rotation update, barriers) then overlap the others' passes instead of idling the SM, and there is no second
      // wave whose stragglers run alone.  Measured on 592 cfg-A pairs per step: 38.8 ms against 41.8 ms with
      // 512-thread CTAs in two waves.  (Caching the points instead of the line vectors was measured and dropped:
      // shared-memory gathers of 96 bytes per line vector cost more than the coalesced stream.)
      if (n_active > 2 * sm_count()) return launch_gnc_nc<1, 128, 4>(st, d_jobs, n_jobs, cap_per_cta);
      if (n_active > sm_count()) return launch_gnc_nc<1, 256, 2>(st, d_jobs, n_jobs, cap_per_cta);
      return launch_gnc_nc<1, 512, 1>(st, d_jobs, n_jobs, cap_per_cta);
    }
    default: return fail(PSULVSB_ERR_INVALID, "launch_gnc_tls: cluster must be 1, 2, 4, 8 or (grid mode) more");
  }
}

int launch_kabsch_batch(cudaStream_t st, const double* src, const double* dst, const uint2* edges,
                        const uint32_t* sets, int k, unsigned long long n_hyp, double* R, double* t) {
  if (n_hyp == 0) return PSULVSB_OK;
  if (k < 1) return fail(PSULVSB_ERR_INVALID, "kabsch_batch: k < 1");
  const unsigned long long threads = n_hyp * 32ull;
  kabsch_batch_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(src, dst, edges, sets, k, n_hyp, R, t);
  PSU_CHECK_LAUNCH("kabsch_batch_kernel");
  return PSULVSB_OK;
}

}  // namespace psulvsb
