// k4_score.cu -- stage 4: fused transform + score + argmax, plus the single-hypothesis FP64 scorer
// and the stand-alone max-stabbing translation kernel.
//
// Reference: the three scoring loops of solve(), registration.cc:1303-1311, :1329-1336 (sampled
// points) and :1417-1444 (all M points): count_j [ | q_j - s (R p_j + t) | <= tau ].
//
// score_batch_kernel: a thread owns HPT hypotheses (s*R, s*t' in registers), the CTA streams its slice of the
// correspondences through shared memory in double-buffered tiles staged by 1-D TMA bulk copies, so a
// thread finishes with the complete inlier count of its hypotheses: no cross-thread reduction of
// counts, only a warp-shuffle / block / grid argmax of (count, hypothesis) packed in 64 bits.
// Packed FP32 (FFMA2): two POINTS travel in the halves of a 64-bit register pair -- the tiles are pair-interleaved
// (common.cuh il_store), so one LDS.128 delivers the same coordinate of points (2q, 2q + 1) as an aligned pair --
// and the hypothesis values enter as scalar broadcasts.  A point pair's coordinate is then the 64-bit operand of the
// 12 consecutive FFMA2 of a thread's 4 hypotheses x 3 rows, which keeps it in the operand-reuse cache: measured
// (profiles/tools/fp32_pipe_probe.cu) 0.99 of the FP32 peak against 0.92 when the shared operand is the 32-bit scalar
// (hypotheses packed, r1), and the band tracking is one three-input FMNMX3 per two units instead of two FMNMX.
// FP32 evaluation on centred coordinates; u = |d|^2 - tau^2 is accumulated with its sign, and a
// hypothesis with any point inside the FP32 error band of the threshold is re-scored exactly: the
// borderline points are re-evaluated in FP64 with the reference's formula (counted).
#include <cuda_runtime.h>

#include "common.cuh"
#include "engine.cuh"
#include "solve_dev.cuh"

namespace psulvsb {

namespace {

constexpr int SB_THREADS = 256;
constexpr int SB_HPT = 4;    // hypotheses per thread
constexpr int SB_TP = 512;   // points per smem tile (2 stages x 2 arrays x 8 KB static smem)

// (packed FP32 helpers fma2 / bc2: common.cuh)
struct ScoreArgs {
  double scale, tau;
  double csrc[3], cdst[3];  // centres the float4 tiles were packed with
  float coord_bound;
};

__global__ void __launch_bounds__(SB_THREADS)
    score_batch_kernel(const float4* __restrict__ srcf, const float4* __restrict__ dstf,  // pair-interleaved records
                       const double* __restrict__ src64, const double* __restrict__ dst64, int n,
                       const double* __restrict__ hyp, unsigned long long n_hyp, unsigned long long hyp_begin,
                       ScoreArgs a, int chunk_points, uint32_t* __restrict__ counts,
                       unsigned long long* __restrict__ border_count, unsigned int* __restrict__ tickets,
                       unsigned long long* __restrict__ best) {
  __shared__ __align__(128) float4 ps[2][SB_TP];
  __shared__ __align__(128) float4 qs[2][SB_TP];
  __shared__ __align__(8) uint64_t bar[2];
  const int tid = threadIdx.x, lane = tid & 31;
  // this CTA's slice of the correspondences (grid.y): many short CTAs instead of a few long ones
  const int p_lo = blockIdx.y * chunk_points;
  const int p_hi = min(n, p_lo + chunk_points);
  if (p_lo >= p_hi) return;
  const int np_chunk = p_hi - p_lo;
  const unsigned long long h0 = ((unsigned long long)blockIdx.x * SB_THREADS + tid) * SB_HPT;

  // ---- hypotheses -> registers: Rf = s R, tf = s (R c_src + t) - c_dst  (centred coordinates)
  float Rf[SB_HPT][9], tf[SB_HPT][3], eps[SB_HPT], mn[SB_HPT];
  int cnt[SB_HPT];
  const double tau2d = a.tau * a.tau;
  const float tau2 = (float)tau2d;
#pragma unroll
  for (int k = 0; k < SB_HPT; ++k) {
    const unsigned long long h = h0 + k;
    cnt[k] = 0;
    mn[k] = 3.0e38f;
    if (h < n_hyp) {
      const double* H = hyp + h * 12;
      double tmax = 0.0;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const double r0 = H[0 * 3 + r], r1 = H[1 * 3 + r], r2 = H[2 * 3 + r];  // column-major R
        Rf[k][r * 3 + 0] = (float)(a.scale * r0);
        Rf[k][r * 3 + 1] = (float)(a.scale * r1);
        Rf[k][r * 3 + 2] = (float)(a.scale * r2);
        const double tp = a.scale * (r0 * a.csrc[0] + r1 * a.csrc[1] + r2 * a.csrc[2] + H[9 + r]) - a.cdst[r];
        tf[k][r] = (float)tp;
        tmax = fmax(tmax, fabs(tp));
      }
      // a wrong fast sign has |u| <= 64 mu tau (G + tau) + 640 (mu G)^2,  G = |t'|_inf + (1 + sqrt3 s) Cmax
      // (DESIGN.md "K4 error band"); tau^2 or the band beyond FP32: eps = inf sends every point to the FP64 fix-up
      const double G = tmax + (1.0 + 1.7320508 * fabs(a.scale)) * (double)a.coord_bound;
      const double muG = 5.9604644775390625e-08 * G;
      const double e = (64.0 * 5.9604644775390625e-08 * a.tau * (G + a.tau) + 640.0 * (muG * muG)) * 1.0001;
      eps[k] = (e < 3.4028234663852886e38 && tau2d < 3.4028234663852886e38) ? (float)e + 1e-37f : __int_as_float(0x7f800000);
    } else {
#pragma unroll
      for (int i = 0; i < 9; ++i) Rf[k][i] = 0.f;
      tf[k][0] = tf[k][1] = tf[k][2] = 0.f;
      eps[k] = 0.f;
    }
  }

  const int ntiles = (np_chunk + SB_TP - 1) / SB_TP;
  if (tid == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  auto issue = [&](int tile) {
    const int st = tile & 1;
    const int p0 = p_lo + tile * SB_TP;
    // whole point pairs (an odd n ends with a zero record that is never scored)
    const uint32_t bytes = (uint32_t)min(SB_TP, (int)il_records((size_t)p_hi) - p0) * (uint32_t)sizeof(float4);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(&bar[st], 2 * bytes);
    tma_load_1d(ps[st], srcf + p0, bytes, &bar[st]);
    tma_load_1d(qs[st], dstf + p0, bytes, &bar[st]);
  };
  if (tid == 0) {
    issue(0);
    if (ntiles > 1) issue(1);
  }
  for (int tile = 0; tile < ntiles; ++tile) {
    const int st = tile & 1;
    mbar_wait(&bar[st], (tile >> 1) & 1);
    const int np = min(SB_TP, np_chunk - tile * SB_TP);
    const int npairs = np >> 1;
#pragma unroll 2
    for (int q = 0; q < npairs; ++q) {
      const float4 pa = ps[st][2 * q], pb = ps[st][2 * q + 1];  // (x0 x1 y0 y1) (z0 z1 . .)
      const float4 qa = qs[st][2 * q], qb = qs[st][2 * q + 1];
      const float2 PX = make_float2(pa.x, pa.y), PY = make_float2(pa.z, pa.w), PZ = make_float2(pb.x, pb.y);
      const float2 QX = make_float2(qa.x, qa.y), QY = make_float2(qa.z, qa.w), QZ = make_float2(qb.x, qb.y);
      // every half is the IEEE result of the scalar chain the fix-up below re-evaluates: tf - q as fma(q, -1, tf) (one
      // rounding: the FADD's value), then z, y, x
#pragma unroll
      for (int k = 0; k < SB_HPT; ++k) {
        const float2 e0 = fma2(QX, bc2(-1.f), bc2(tf[k][0]));
        const float2 e1 = fma2(QY, bc2(-1.f), bc2(tf[k][1]));
        const float2 e2 = fma2(QZ, bc2(-1.f), bc2(tf[k][2]));
        const float2 d0 = fma2(bc2(Rf[k][0]), PX, fma2(bc2(Rf[k][1]), PY, fma2(bc2(Rf[k][2]), PZ, e0)));
        const float2 d1 = fma2(bc2(Rf[k][3]), PX, fma2(bc2(Rf[k][4]), PY, fma2(bc2(Rf[k][5]), PZ, e1)));
        const float2 d2 = fma2(bc2(Rf[k][6]), PX, fma2(bc2(Rf[k][7]), PY, fma2(bc2(Rf[k][8]), PZ, e2)));
        const float2 u = fma2(d2, d2, fma2(d1, d1, fma2(d0, d0, bc2(-tau2))));
        cnt[k] += (int)(__float_as_uint(u.x) >> 31);
        cnt[k] += (int)(__float_as_uint(u.y) >> 31);
        mn[k] = fminf(mn[k], fminf(fabsf(u.x), fabsf(u.y)));
      }
    }
    if (np & 1) {  // the last point of an odd n
      const float4 p = il_load(ps[st], np - 1);
      const float4 q = il_load(qs[st], np - 1);
#pragma unroll
      for (int k = 0; k < SB_HPT; ++k) {
        const float d0 = fmaf(Rf[k][0], p.x, fmaf(Rf[k][1], p.y, fmaf(Rf[k][2], p.z, fmaf(q.x, -1.f, tf[k][0]))));
        const float d1 = fmaf(Rf[k][3], p.x, fmaf(Rf[k][4], p.y, fmaf(Rf[k][5], p.z, fmaf(q.y, -1.f, tf[k][1]))));
        const float d2 = fmaf(Rf[k][6], p.x, fmaf(Rf[k][7], p.y, fmaf(Rf[k][8], p.z, fmaf(q.z, -1.f, tf[k][2]))));
        const float u = fmaf(d2, d2, fmaf(d1, d1, fmaf(d0, d0, -tau2)));
        cnt[k] += (int)(__float_as_uint(u) >> 31);
        mn[k] = fminf(mn[k], fabsf(u));
      }
    }
    __syncthreads();  // everyone is done with stage st
    if (tid == 0 && tile + 2 < ntiles) issue(tile + 2);
  }

  // ---- exact fix-up for hypotheses with a point inside the band (rare)
  unsigned int nborder = 0;
#pragma unroll
  for (int k = 0; k < SB_HPT; ++k) {
    const unsigned long long h = h0 + k;
    if (h < n_hyp && !(mn[k] > eps[k])) {
      const double* H = hyp + h * 12;
      double R[9], t[3];
      for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) R[r * 3 + c] = H[c * 3 + r];
        t[r] = H[9 + r];
      }
      for (int j = p_lo; j < p_hi; ++j) {
        const float4 p = il_load(srcf, j);
        const float4 q = il_load(dstf, j);
        const float d0 = fmaf(Rf[k][0], p.x, fmaf(Rf[k][1], p.y, fmaf(Rf[k][2], p.z, tf[k][0] - q.x)));
        const float d1 = fmaf(Rf[k][3], p.x, fmaf(Rf[k][4], p.y, fmaf(Rf[k][5], p.z, tf[k][1] - q.y)));
        const float d2 = fmaf(Rf[k][6], p.x, fmaf(Rf[k][7], p.y, fmaf(Rf[k][8], p.z, tf[k][2] - q.z)));
        const float u = fmaf(d2, d2, fmaf(d1, d1, fmaf(d0, d0, -tau2)));
        if (!(fabsf(u) > eps[k])) {
          ++nborder;
          const bool fast_in = (__float_as_uint(u) >> 31) != 0u;
          const bool exact_in = residual_ref(src64 + 3 * (size_t)j, dst64 + 3 * (size_t)j, a.scale, R, t) <= a.tau;
          cnt[k] += (exact_in ? 1 : 0) - (fast_in ? 1 : 0);
        }
      }
    }
  }

  // ---- outputs: this chunk's contribution to the counts (the argmax runs once all chunks are in)
#pragma unroll
  for (int k = 0; k < SB_HPT; ++k) {
    const unsigned long long h = h0 + k;
    if (h < n_hyp && cnt[k] != 0) atomicAdd(&counts[h], (uint32_t)cnt[k]);
  }
  const unsigned int nb = (unsigned int)warp_sum_int((int)nborder);
  if (lane == 0 && nb && border_count) atomicAdd(border_count, (unsigned long long)nb);

  // ---- argmax, fused: the CTA that completes a hypothesis group (the last of its gridDim.y correspondence slices to
  // add its counts) reduces the group's keys (count << 32 | ~id: the first best hypothesis wins, as the strict '>' of
  // registration.cc:1337) warp -> block and issues ONE atomicMax.  With a single slice the counts never leave the
  // registers before the reduction.
  if (best == nullptr) return;
  __shared__ int is_last;
  __shared__ unsigned long long warp_best[SB_THREADS / 32];
  if (gridDim.y > 1) {
    __threadfence();  // this CTA's atomicAdds are visible before its ticket
    __syncthreads();
    if (tid == 0) is_last = (atomicAdd(&tickets[blockIdx.x], 1u) == gridDim.y - 1u) ? 1 : 0;
    __syncthreads();
    if (!is_last) return;
    __threadfence();
  }
  unsigned long long mybest = 0ull;
#pragma unroll
  for (int k = 0; k < SB_HPT; ++k) {
    const unsigned long long h = h0 + k;
    if (h < n_hyp) {
      const uint32_t c = (gridDim.y > 1) ? __ldcg(&counts[h]) : (uint32_t)cnt[k];
      const unsigned long long key = ((unsigned long long)c << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)(hyp_begin + h));
      mybest = key > mybest ? key : mybest;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long x = __shfl_xor_sync(0xffffffffu, mybest, o);
    mybest = x > mybest ? x : mybest;
  }
  if (lane == 0) warp_best[tid >> 5] = mybest;
  __syncthreads();
  if (tid == 0) {
    unsigned long long b = warp_best[0];
#pragma unroll
    for (int w = 1; w < SB_THREADS / 32; ++w) b = warp_best[w] > b ? warp_best[w] : b;
    if (b) atomicMax(best, b);
  }
}

// n = 0: the key of the first hypothesis (count 0), combined like the batch kernel's
__global__ void score_empty_best_kernel(unsigned long long* __restrict__ best, unsigned long long key) {
  if (key) atomicMax(best, key);
}

// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    score_one_kernel(const double* __restrict__ src, const double* __restrict__ dst, int n, double scale,
                     const double* __restrict__ Rcm, const double* __restrict__ tt, double tau,
                     uint8_t* __restrict__ inliers, double* __restrict__ residuals, int* __restrict__ count) {
  double R[9], t[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c) R[r * 3 + c] = Rcm[c * 3 + r];
    t[r] = tt[r];
  }
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  bool in = false;
  if (j < n) {
    const double res = residual_ref(src + 3 * (size_t)j, dst + 3 * (size_t)j, scale, R, t);
    in = res <= tau;
    if (inliers) inliers[j] = in ? 1 : 0;
    if (residuals) residuals[j] = res;
  }
  // warp popc reduction of the predicate
  const unsigned int bal = __ballot_sync(0xffffffffu, in);
  if ((threadIdx.x & 31) == 0 && bal && count) atomicAdd(count, __popc(bal));
}

// stand-alone translation stage: compact the flagged points (ascending), then block_translation
__global__ void __launch_bounds__(BLK)
    tls_translation_kernel(const double* __restrict__ src, const double* __restrict__ dst,
                           const uint8_t* __restrict__ flags, int n, double scale, const double* __restrict__ Rcm,
                           double sigma, const double* __restrict__ last_best, int* __restrict__ idx,
                           double* __restrict__ xs, double* __restrict__ sorted, double* __restrict__ t_out,
                           int* __restrict__ n_points) {
  __shared__ BlockScratch scratch;
  __shared__ int base_s;
  const int tid = threadIdx.x;
  if (tid == 0) base_s = 0;
  __syncthreads();
  for (int j0 = 0; j0 < n; j0 += BLK) {
    const int j = j0 + tid;
    const int f = (j < n && flags[j]) ? 1 : 0;
    int ea, eb, ta, tb;
    block_scan2(&scratch, f, 0, ea, eb, ta, tb);
    const int base = base_s;
    if (f) idx[base + ea] = j;
    __syncthreads();
    if (tid == 0) base_s = base + ta;
    __syncthreads();
  }
  const int P = base_s;
  double R[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) R[r * 3 + c] = Rcm[c * 3 + r];
  double t[3] = {0.0, 0.0, 0.0};
  double lb[3];
  if (last_best) {
    lb[0] = last_best[0];
    lb[1] = last_best[1];
    lb[2] = last_best[2];
  }
  block_translation(&scratch, src, dst, idx, P, scale, R, sigma, last_best ? lb : nullptr, xs, t, sorted);
  if (tid == 0) {
    t_out[0] = t[0];
    t_out[1] = t[1];
    t_out[2] = t[2];
    if (n_points) *n_points = P;
  }
}

}  // namespace

int launch_score_batch(cudaStream_t st, const float4* src, const float4* dst, const double* src64, const double* dst64,
                       int n, const double* hyp, unsigned long long n_hyp, unsigned long long hyp_begin, double scale,
                       double tau, double coord_bound, const double* csrc, const double* cdst, uint32_t* counts,
                       unsigned long long* best, unsigned long long* border) {
  if (n < 0) return fail(PSULVSB_ERR_INVALID, "score_batch: n < 0");
  if (n_hyp == 0) return PSULVSB_OK;
  // ids hyp_begin .. hyp_begin + n_hyp - 1 must stay below 0xFFFFFFFF (written so that it cannot wrap)
  if (n_hyp > 0xFFFFFFFFull || hyp_begin > 0xFFFFFFFFull - n_hyp)
    return fail(PSULVSB_ERR_UNSUPPORTED, "score_batch: hypothesis id > 32 bits");
  if (n == 0) {  // no points: every count is 0, and the first hypothesis is the best
    PSU_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * n_hyp, st));
    if (best) {
      score_empty_best_kernel<<<1, 1, 0, st>>>(best, 0xFFFFFFFFull - hyp_begin);
      PSU_CHECK_LAUNCH("score_empty_best_kernel");
    }
    return PSULVSB_OK;
  }
  ScoreArgs a;
  a.scale = scale;
  a.tau = tau;
  for (int r = 0; r < 3; ++r) {
    a.csrc[r] = csrc ? csrc[r] : 0.0;
    a.cdst[r] = cdst ? cdst[r] : 0.0;
  }
  a.coord_bound = (float)(coord_bound * 1.0000002);
  const unsigned long long per_cta = (unsigned long long)SB_THREADS * SB_HPT;
  const unsigned long long gx = (n_hyp + per_cta - 1) / per_cta;
  // slice the correspondences too (grid.y): slices of >= 4 tiles, preferably >= 10 waves of 2 CTAs per SM; among
  // the admissible slice lengths take the one that fills its last wave best (2^20 hypotheses x 50 000 points in three
  // slices of 8 tiles are 10.4 waves: the eleventh runs a third full, 6 % of the sweep)
  const unsigned long long slots = (unsigned long long)sm_count() * 2ull;
  const int n_tiles = (n + SB_TP - 1) / SB_TP;
  int best_tiles = n_tiles;
  double best_eff = -1.0;
  const int t_min = n_tiles < 4 ? n_tiles : 4;  // a slice amortises its CTA's prologue (48 doubles per thread) over >= 4 tiles
  for (int t = n_tiles; t >= t_min; --t) {       // tiles per slice, long slices first (ties keep the longer)
    const unsigned long long gy_t = (unsigned long long)((n_tiles + t - 1) / t);
    if (gy_t > 65535ull) break;
    const unsigned long long ctas = gx * gy_t;
    const unsigned long long waves = (ctas + slots - 1) / slots;
    double eff = (double)ctas / (double)(waves * slots);
    if (waves < 10) eff *= 0.5 + 0.05 * (double)waves;  // few waves: the last CTAs' length weighs more than the fill
    if (eff > best_eff + 1e-9) {
      best_eff = eff;
      best_tiles = t;
    }
  }
  const int chunk_points = best_tiles * SB_TP;  // tile-aligned: every bulk copy stays 16-byte aligned
  const unsigned gy = (unsigned)((n + chunk_points - 1) / chunk_points);
  // the kernel streams pair-interleaved records (common.cuh il_store), built here from the caller's per-point ones
  struct AsyncScratch {  // stream-ordered scratch, returned on every path out of this function
    void* p = nullptr;
    cudaStream_t s;
    explicit AsyncScratch(cudaStream_t st_) : s(st_) {}
    ~AsyncScratch() {
      if (p) cudaFreeAsync(p, s);
    }
  } il_mem(st), ticket_mem(st);
  const size_t nrec = il_records((size_t)n);
  PSU_CUDA(cudaMallocAsync(&il_mem.p, sizeof(float4) * 2 * nrec, st));
  float4* il = static_cast<float4*>(il_mem.p);
  if (int rc = launch_interleave_points(st, src, n, il)) return rc;
  if (int rc = launch_interleave_points(st, dst, n, il + nrec)) return rc;
  PSU_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * n_hyp, st));
  unsigned int* tickets = nullptr;  // one "slices done" counter per hypothesis group (stream-ordered scratch)
  if (best && gy > 1) {
    PSU_CUDA(cudaMallocAsync(&ticket_mem.p, sizeof(unsigned int) * gx, st));
    tickets = static_cast<unsigned int*>(ticket_mem.p);
    PSU_CUDA(cudaMemsetAsync(tickets, 0, sizeof(unsigned int) * gx, st));
  }
  score_batch_kernel<<<dim3((unsigned)gx, gy), SB_THREADS, 0, st>>>(il, il + nrec, src64, dst64, n, hyp, n_hyp, hyp_begin, a,
                                                                     chunk_points, counts, border, tickets, best);
  const cudaError_t le = cudaGetLastError();
  if (le != cudaSuccess) return fail(PSULVSB_ERR_CUDA, std::string("score_batch_kernel launch: ") + cudaGetErrorString(le));
  return PSULVSB_OK;
}

int launch_score_one(cudaStream_t st, const double* src, const double* dst, int n, double scale, const double* R,
                     const double* t, double tau, uint8_t* inliers, double* residuals, int* count) {
  if (n <= 0) return PSULVSB_OK;
  score_one_kernel<<<(n + 255) / 256, 256, 0, st>>>(src, dst, n, scale, R, t, tau, inliers, residuals, count);
  PSU_CHECK_LAUNCH("score_one_kernel");
  return PSULVSB_OK;
}

int launch_tls_translation(cudaStream_t st, const double* src, const double* dst, const uint8_t* flags, int n,
                           double scale, const double* R, double noise, const double* last_best, double* t_out,
                           int* n_points) {
  if (n <= 0) return fail(PSULVSB_ERR_INVALID, "tls_translation: n <= 0");
  int* idx = nullptr;
  double* xs = nullptr;
  PSU_CUDA(cudaMallocAsync((void**)&idx, sizeof(int) * (size_t)n, st));
  PSU_CUDA(cudaMallocAsync((void**)&xs, sizeof(double) * (3 * ((size_t)n + 1) + translation_sort_doubles(n)), st));
  tls_translation_kernel<<<1, BLK, 0, st>>>(src, dst, flags, n, scale, R, noise, last_best, idx, xs,
                                            xs + 3 * ((size_t)n + 1), t_out, n_points);
  cudaError_t e = cudaGetLastError();
  cudaFreeAsync(idx, st);
  cudaFreeAsync(xs, st);
  if (e != cudaSuccess) return fail(PSULVSB_ERR_CUDA, std::string("tls_translation_kernel launch: ") + cudaGetErrorString(e));
  return PSULVSB_OK;
}

}  // namespace psulvsb
