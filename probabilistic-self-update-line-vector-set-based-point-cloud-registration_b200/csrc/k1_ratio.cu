// k1_ratio.cu -- stage 1 for the unknown-scale configuration (Params::estimate_scaling = true):
// the length-RATIO histogram and its reduced set (registration.cc:687-752).
//
// The reference pushes every line vector l = (i < j) into bin floor(X / MaxScale * H.size()) of a
// 200 000-bin histogram, X = |t_j - t_i| / |s_j - s_i|, remembers the first bin to reach the running
// maximum height, and takes as reduced set the members of the bins {peak, peak - 1, peak + 1}, each
// in line-vector order, concatenated in that order (registration.cc:744-752).
//
// Here (all FP64, reference operation order, so bins are bit-identical):
//   ratio_bins_kernel : bin of every pair -> pair_bin[l] (row-major pair order) + histogram
//                       (shared-memory privatised for bins < 2048, global atomics beyond)
//   peak kernels      : max height; among the bins at that height the one whose LAST member comes
//                       first in pair order is "the first to reach it" (strict '>' at :725)
//   class count / scan / emit : ordered compaction of the three bins into endpoint pairs
// A ratio above MaxScale (10000 at first) makes the reference grow MaxScale and the histogram in the middle of its pair
// loop (:714-718), which changes the bin of every LATER pair.  That is reproduced without a candidate list: growth at
// pair l needs X_l > MaxScale, and MaxScale <- ceil(MaxScale + X) more than doubles it, so at most
// RATIO_MAX_GROWTHS growths keep MaxScale <= RATIO_MAX_SCALE.  A first pass stores the largest ratio of every row
// (fmax: a 0 / 0 NaN never grows anything); one CTA then replays the growth rule, jumping to the first row whose
// maximum exceeds the MaxScale in force and scanning it for the first such pair, and leaves the break points
// (pair index -> MaxScale from there on); the binning pass looks its MaxScale up in that list.  Only an infinite
// ratio (coincident source points with distinct targets: undefined behaviour in the reference) or a final MaxScale
// beyond RATIO_MAX_SCALE is refused (PSULVSB_ERR_UNSUPPORTED).
#include <cuda_runtime.h>

#include <climits>
#include <functional>
#include <string>
#include <vector>

#include "common.cuh"
#include "engine.cuh"

namespace psulvsb {

namespace {

constexpr int RB_THREADS = 256;
constexpr int RB_SMEM_BINS = 2048;
constexpr double kMaxScale0 = 10000.0;  // registration.cc:688
constexpr double kBinSize = 20.0;       // registration.cc:687

__device__ __forceinline__ unsigned long long row_offset(unsigned long long i, unsigned long long n) {
  return i * (2ull * n - i - 1ull) / 2ull;  // number of pairs (a < b) with a < i
}

__device__ __forceinline__ double pair_ratio(const double* __restrict__ s, const double* __restrict__ t, int i, int j) {
  const double sx = dsub(s[3 * j + 0], s[3 * i + 0]), sy = dsub(s[3 * j + 1], s[3 * i + 1]),
               sz = dsub(s[3 * j + 2], s[3 * i + 2]);
  const double tx = dsub(t[3 * j + 0], t[3 * i + 0]), ty = dsub(t[3 * j + 1], t[3 * i + 1]),
               tz = dsub(t[3 * j + 2], t[3 * i + 2]);
  return sqrt(sqnorm3(tx, ty, tz)) / sqrt(sqnorm3(sx, sy, sz));
}

// MaxScale in force when pair l is binned: the last break point at or before l (growth precedes the binning
// of the pair that triggers it, registration.cc:714-723)
__device__ __forceinline__ double scale_at(const RatioJob& job, unsigned long long l) {
  const unsigned int nbp = *job.bp_n;
  double ms = kMaxScale0;
  for (unsigned int k = 0; k < nbp; ++k) {  // a handful of entries at most
    if (job.bp_idx[k] <= l) ms = job.bp_scale[k];
  }
  return ms;
}

// registration.cc:697-723 for one pair, FP64 in the reference's operation order
__device__ __forceinline__ uint32_t ratio_bin(double X, double max_scale) {
  const double hsize = dmul(max_scale, kBinSize);  // H.size() == MaxScale * binsize, exact (both integers)
  const double f = floor(dmul(X / max_scale, hsize));
  long long h = (f == f && fabs(f) < 9.0e18) ? (long long)f : 0ll;  // NaN (0 / 0): the reference files it under bin 0
  if (h == (long long)hsize)
    h -= 1;
  else if (h > (long long)hsize || h < 0)
    h = 0;
  return (uint32_t)h;
}

// pass 0: the largest ratio of every row (fmax ignores the NaN of 0 / 0; an infinite ratio stays infinite)
__global__ void __launch_bounds__(RB_THREADS) ratio_rowmax_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.y];
  if (!job.active) return;
  const int n = job.n;
  const int i = blockIdx.x;
  if (i >= n - 1) return;
  __shared__ double wmax[RB_THREADS / 32];
  double m = 0.0;
  for (int j = i + 1 + threadIdx.x; j < n; j += RB_THREADS) m = fmax(m, pair_ratio(job.src64, job.dst64, i, j));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < RB_THREADS / 32; ++w) m = fmax(m, wmax[w]);
    job.row_max[i] = m;
  }
}

constexpr int RG_THREADS = 1024;

__device__ __forceinline__ int block_min(int v, int* s) {
  if (threadIdx.x == 0) *s = INT_MAX;
  __syncthreads();
  if (v != INT_MAX) atomicMin(s, v);
  __syncthreads();
  v = *s;
  __syncthreads();
  return v;
}

// one CTA per job replays registration.cc:714-718 in pair order: the first pair at or after (r, j0) whose ratio exceeds
// the MaxScale in force is searched in row r, else in the first later row whose maximum exceeds it
__global__ void __launch_bounds__(RG_THREADS) ratio_growth_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.x];
  if (!job.active) return;
  __shared__ int s_min;
  const int n = job.n, rows = n - 1;
  bool inf = false;
  for (int r = threadIdx.x; r < rows; r += RG_THREADS) inf |= isinf(job.row_max[r]);
  if (__syncthreads_or(inf)) {  // ceil(MaxScale + inf) is undefined behaviour in the reference
    if (threadIdx.x == 0) {
      *job.bp_n = 0u;
      *job.final_scale = kMaxScale0;
      *job.bad = 1;
    }
    return;
  }
  double cur = kMaxScale0;
  unsigned int nbp = 0;
  int r = 0, j0 = 1;
  while (r < rows && cur <= RATIO_MAX_SCALE) {
    int jm = INT_MAX;
    for (int j = j0 + threadIdx.x; j < n; j += RG_THREADS)
      if (pair_ratio(job.src64, job.dst64, r, j) > cur) {
        jm = j;  // each thread walks its j ascending: its first hit is its smallest
        break;
      }
    jm = block_min(jm, &s_min);
    if (jm == INT_MAX) {
      int rm = INT_MAX;
      for (int q = r + 1 + threadIdx.x; q < rows; q += RG_THREADS)
        if (job.row_max[q] > cur) {
          rm = q;
          break;
        }
      rm = block_min(rm, &s_min);
      if (rm == INT_MAX) break;
      r = rm;
      j0 = rm + 1;
      continue;
    }
    cur = ceil(dadd(cur, pair_ratio(job.src64, job.dst64, r, jm)));
    if (threadIdx.x == 0) {
      job.bp_idx[nbp] = row_offset((unsigned long long)r, (unsigned long long)n) + (unsigned long long)(jm - r - 1);
      job.bp_scale[nbp] = cur;
    }
    ++nbp;
    j0 = jm + 1;
  }
  if (threadIdx.x == 0) {
    *job.bp_n = nbp;
    *job.final_scale = cur;
    *job.bad = cur > RATIO_MAX_SCALE ? 3 : 0;
  }
}

__global__ void __launch_bounds__(RB_THREADS) ratio_bins_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.y];
  if (!job.active) return;
  const int n = job.n;
  const int i = blockIdx.x;
  if (i >= n - 1) return;
  __shared__ unsigned int sh[RB_SMEM_BINS];
  for (int k = threadIdx.x; k < RB_SMEM_BINS; k += RB_THREADS) sh[k] = 0u;
  __syncthreads();
  const unsigned long long base = row_offset((unsigned long long)i, (unsigned long long)n);
  const bool grown = *job.bp_n != 0u;
  for (int j = i + 1 + threadIdx.x; j < n; j += RB_THREADS) {
    const unsigned long long l = base + (unsigned long long)(j - i - 1);
    const double X = pair_ratio(job.src64, job.dst64, i, j);
    const uint32_t b = ratio_bin(X, grown ? scale_at(job, l) : kMaxScale0);
    job.pair_bin[l] = b;
    if (b < RB_SMEM_BINS)
      atomicAdd(&sh[b], 1u);
    else
      atomicAdd(&job.hist[b], 1u);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < RB_SMEM_BINS; k += RB_THREADS)
    if (sh[k]) atomicAdd(&job.hist[k], sh[k]);
}

// max height over the histogram (one CTA per job)
__global__ void __launch_bounds__(1024) ratio_max_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.x];
  if (!job.active) return;
  __shared__ unsigned int wmax[32];
  unsigned int m = 0;
  const long long hsize = (long long)(*job.final_scale * kBinSize);
  for (long long b = threadIdx.x; b < hsize; b += 1024) m = max(m, job.hist[b]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int mm = 0;
    for (int w = 0; w < 32; ++w) mm = max(mm, wmax[w]);
    job.peak[0] = mm;          // max height
    job.peak[1] = 0xFFFFFFFFu; // peak bin (filled by ratio_peak_kernel)
  }
}

// position (pair index) of the last member of every bin at the max height
__global__ void __launch_bounds__(RB_THREADS) ratio_last_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.y];
  if (!job.active) return;
  const unsigned long long L = (unsigned long long)job.n * (unsigned long long)(job.n - 1) / 2ull;
  const unsigned int mh = job.peak[0];
  for (unsigned long long l = (unsigned long long)blockIdx.x * RB_THREADS + threadIdx.x; l < L;
       l += (unsigned long long)gridDim.x * RB_THREADS) {
    const uint32_t b = job.pair_bin[l];
    if (job.hist[b] == mh) atomicMax(&job.last[b], l + 1ull);
  }
}

// the bin at max height whose last member comes first ("first to reach the running maximum")
__global__ void __launch_bounds__(1024) ratio_peak_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.x];
  if (!job.active) return;
  __shared__ unsigned long long wbest[32];
  __shared__ unsigned int wbin[32];
  const unsigned int mh = job.peak[0];
  unsigned long long best = ~0ull;
  unsigned int bin = 0xFFFFFFFFu;
  const long long hsize = (long long)(*job.final_scale * kBinSize);
  for (long long b = threadIdx.x; b < hsize; b += 1024)
    if (job.hist[b] == mh && mh > 0) {
      const unsigned long long last = job.last[b];
      if (last < best) {
        best = last;
        bin = (unsigned int)b;
      }
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long ob = __shfl_xor_sync(0xffffffffu, best, o);
    const unsigned int obin = __shfl_xor_sync(0xffffffffu, bin, o);
    if (ob < best) {
      best = ob;
      bin = obin;
    }
  }
  if ((threadIdx.x & 31) == 0) {
    wbest[threadIdx.x >> 5] = best;
    wbin[threadIdx.x >> 5] = bin;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 0; w < 32; ++w)
      if (wbest[w] < best) {
        best = wbest[w];
        bin = wbin[w];
      }
    job.peak[1] = bin;
  }
}

// class of a bin w.r.t. the peak: 0 = peak, 1 = peak - 1, 2 = peak + 1 (registration.cc:746-750), 3 = none
__device__ __forceinline__ int bin_class(uint32_t b, uint32_t peak, uint32_t hsize) {
  if (b == peak) return 0;
  if (peak != 0u && b == peak - 1u) return 1;
  if (peak != hsize - 1u && b == peak + 1u) return 2;
  return 3;
}

// one warp per row: members of each class in the row -> class_counts[c * n + i]
__global__ void __launch_bounds__(256) ratio_class_count_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.y];
  if (!job.active) return;
  const int n = job.n;
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const uint32_t peak = job.peak[1];
  const uint32_t hsize = (uint32_t)(*job.final_scale * kBinSize);
  unsigned int c0 = 0, c1 = 0, c2 = 0;
  if (row < n - 1 && peak != 0xFFFFFFFFu) {
    const unsigned long long base = row_offset((unsigned long long)row, (unsigned long long)n);
    const int len = n - 1 - row;
    for (int k = lane; k < len; k += 32) {
      const int c = bin_class(job.pair_bin[base + k], peak, hsize);
      c0 += c == 0;
      c1 += c == 1;
      c2 += c == 2;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    c0 += __shfl_xor_sync(0xffffffffu, c0, o);
    c1 += __shfl_xor_sync(0xffffffffu, c1, o);
    c2 += __shfl_xor_sync(0xffffffffu, c2, o);
  }
  if (lane == 0) {
    job.class_counts[row] = c0;
    job.class_counts[n + row] = c1;
    job.class_counts[2 * n + row] = c2;
  }
}

// exclusive scan over the 3n (class-major) counts -> offsets[3n + 1]; total -> *n_edges
__global__ void __launch_bounds__(1024) ratio_class_scan_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.x];
  if (!job.active) return;
  const int m = 3 * job.n;
  __shared__ unsigned long long part[1024];
  const int tid = threadIdx.x;
  const int per = (m + 1023) / 1024;
  const int lo = min(m, tid * per), hi = min(m, lo + per);
  unsigned long long s = 0;
  for (int i = lo; i < hi; ++i) s += job.class_counts[i];
  part[tid] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    const unsigned long long v = (tid >= off) ? part[tid - off] : 0ull;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  unsigned long long run = part[tid] - s;
  for (int i = lo; i < hi; ++i) {
    job.class_offsets[i] = run;
    run += job.class_counts[i];
  }
  if (tid == 1023) {
    job.class_offsets[m] = part[1023];
    *job.n_edges = part[1023];
  }
}

// one warp per row: emit (i, j) of every member of class c at class_offsets[c * n + i], ascending j, in edge format F
template <class F>
__global__ void __launch_bounds__(256) ratio_class_emit_kernel(const RatioJob* __restrict__ jobs) {
  const RatioJob& job = jobs[blockIdx.y];
  if (!job.active || !job.edges) return;
  const int n = job.n;
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n - 1) return;
  const uint32_t peak = job.peak[1];
  if (peak == 0xFFFFFFFFu) return;
  const uint32_t hsize = (uint32_t)(*job.final_scale * kBinSize);
  const unsigned long long base = row_offset((unsigned long long)row, (unsigned long long)n);
  const int len = n - 1 - row;
  unsigned long long pos[3] = {job.class_offsets[row], job.class_offsets[n + row], job.class_offsets[2 * n + row]};
  for (int k0 = 0; k0 < len; k0 += 32) {
    const int k = k0 + lane;
    const int c = (k < len) ? bin_class(job.pair_bin[base + k], peak, hsize) : 3;
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      const unsigned int m = __ballot_sync(0xffffffffu, c == cc);
      if (c == cc) {
        const unsigned long long p = pos[cc] + (unsigned long long)__popc(m & ((1u << lane) - 1u));
        if (p < job.cap) F::store(job.edges, p, (unsigned)row, (unsigned)(row + 1 + k));
      }
      pos[cc] += (unsigned long long)__popc(m);
    }
  }
}

}  // namespace

// phase 0: row maxima + replay of the growth rule (final MaxScale ready -> host sizes the histogram);
// phase 1: bins + histogram + peak + class counts + scan (n_edges ready); phase 2: emit edges
static int launch_ratio_reduced_set(cudaStream_t st, const RatioJob* d_jobs, int n_jobs, int max_n, int phase,
                                    bool narrow = false) {
  if (n_jobs <= 0 || max_n < 2) return PSULVSB_OK;
  const long long row_threads = (long long)max_n * 32;
  const dim3 row_grid((unsigned)((row_threads + 255) / 256), (unsigned)n_jobs);
  if (phase == 0) {
    ratio_rowmax_kernel<<<dim3((unsigned)(max_n - 1), (unsigned)n_jobs), RB_THREADS, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_rowmax_kernel");
    ratio_growth_kernel<<<n_jobs, RG_THREADS, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_growth_kernel");
  } else if (phase == 1) {
    ratio_bins_kernel<<<dim3((unsigned)(max_n - 1), (unsigned)n_jobs), RB_THREADS, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_bins_kernel");
    ratio_max_kernel<<<n_jobs, 1024, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_max_kernel");
    const unsigned long long L = (unsigned long long)max_n * (unsigned long long)(max_n - 1) / 2ull;
    unsigned long long gx = (L + RB_THREADS * 8 - 1) / (RB_THREADS * 8);
    if (gx > sm_count() * 16) gx = sm_count() * 16;
    if (gx < 1) gx = 1;
    ratio_last_kernel<<<dim3((unsigned)gx, (unsigned)n_jobs), RB_THREADS, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_last_kernel");
    ratio_peak_kernel<<<n_jobs, 1024, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_peak_kernel");
    ratio_class_count_kernel<<<row_grid, 256, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_class_count_kernel");
    ratio_class_scan_kernel<<<n_jobs, 1024, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_class_scan_kernel");
  } else {
    if (narrow)
      ratio_class_emit_kernel<EdgeNarrow><<<row_grid, 256, 0, st>>>(d_jobs);
    else
      ratio_class_emit_kernel<EdgeWide><<<row_grid, 256, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("ratio_class_emit_kernel");
  }
  return PSULVSB_OK;
}

int ratio_count(cudaStream_t st, std::vector<RatioJob>& rj, RatioJob* d_rj, int max_n,
                const std::function<void*(size_t)>& hist_arena, cudaEvent_t ev0, cudaEvent_t ev1) {
  const int B = (int)rj.size();
  PSU_CUDA(cudaMemcpyAsync(d_rj, rj.data(), sizeof(RatioJob) * (size_t)B, cudaMemcpyHostToDevice, st));
  if (int rc = launch_ratio_reduced_set(st, d_rj, B, max_n, 0)) return rc;
  std::vector<double> fscale((size_t)B);
  std::vector<int> bad((size_t)B);
  PSU_CUDA(cudaMemcpyAsync(fscale.data(), rj[0].final_scale, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, st));
  PSU_CUDA(cudaMemcpyAsync(bad.data(), rj[0].bad, sizeof(int) * (size_t)B, cudaMemcpyDeviceToHost, st));
  PSU_CUDA(cudaStreamSynchronize(st));
  size_t bins_total = 0;
  for (int b = 0; b < B; ++b) {
    if (bad[(size_t)b])
      return fail(PSULVSB_ERR_UNSUPPORTED,
                  "problem " + std::to_string(b) +
                      (bad[(size_t)b] == 1 ? ": an infinite length ratio (coincident source points with distinct targets; "
                                             "registration.cc:714-718 is undefined there)"
                                           : ": the ratio histogram would outgrow the supported MaxScale of 2e6 "
                                             "(registration.cc:714-718)"));
    bins_total += (size_t)(fscale[(size_t)b] * kBinSize) + 64;
  }
  const size_t bytes = bins_total * (sizeof(unsigned int) + sizeof(unsigned long long));
  char* hb = static_cast<char*>(hist_arena(bytes));
  if (!hb) return PSULVSB_ERR_CUDA;
  size_t off = 0;
  for (int b = 0; b < B; ++b) {
    rj[(size_t)b].last = reinterpret_cast<unsigned long long*>(hb + off);
    off += ((size_t)(fscale[(size_t)b] * kBinSize) + 64) * sizeof(unsigned long long);
  }
  for (int b = 0; b < B; ++b) {
    rj[(size_t)b].hist = reinterpret_cast<unsigned int*>(hb + off);
    off += ((size_t)(fscale[(size_t)b] * kBinSize) + 64) * sizeof(unsigned int);
  }
  PSU_CUDA(cudaMemsetAsync(hb, 0, off, st));
  PSU_CUDA(cudaMemcpyAsync(d_rj, rj.data(), sizeof(RatioJob) * (size_t)B, cudaMemcpyHostToDevice, st));
  if (ev0) PSU_CUDA(cudaEventRecord(ev0, st));
  if (int rc = launch_ratio_reduced_set(st, d_rj, B, max_n, 1)) return rc;
  if (ev1) PSU_CUDA(cudaEventRecord(ev1, st));
  return PSULVSB_OK;
}

int ratio_emit(cudaStream_t st, const std::vector<RatioJob>& rj, RatioJob* d_rj, int max_n, bool narrow) {
  PSU_CUDA(cudaMemcpyAsync(d_rj, rj.data(), sizeof(RatioJob) * rj.size(), cudaMemcpyHostToDevice, st));
  return launch_ratio_reduced_set(st, d_rj, (int)rj.size(), max_n, 2, narrow);
}

}  // namespace psulvsb
