// engine.cu -- host side of the lock-step batch engine: device arenas, problem upload, and the
// launch sequence that replaces RobustRegistrationSolver::solve (registration.cc:622-1535) for a
// batch of B independent registrations on one B200.
//
//   upload : problems -> one pinned staging buffer -> HBM (one copy per element type)
//   solve  : pack float4 tiles -> K1 bit mask (all jobs, one launch) -> row scan -> [n_red to host:
//            sizes the edge arena] -> edge compaction -> init -> ticks until every job is done
//            -> refinement -> solutions to host.
// The only host synchronisations are the n_red read-back and one 4-byte "jobs done" poll per tick.
#include <cuda_runtime.h>
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "common.cuh"
#include "engine.cuh"
#include "engine_kernels.cuh"
#include "engine_state.cuh"

namespace psulvsb {

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return PSULVSB_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      p = nullptr;
      return fail(PSULVSB_ERR_CUDA, std::string("cudaMalloc(") + std::to_string(want) + "): " + cudaGetErrorString(e));
    }
    cap = want;
    return PSULVSB_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return PSULVSB_OK;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e != cudaSuccess) {
      p = nullptr;
      return fail(PSULVSB_ERR_CUDA, std::string("cudaMallocHost: ") + cudaGetErrorString(e));
    }
    cap = want;
    return PSULVSB_OK;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
};

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bump allocator over one arena (sizes first with base == nullptr, then hands out pointers)
struct Bump {
  char* base = nullptr;
  size_t off = 0;
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 128);
    T* r = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return r;
  }
};

struct PackJob {
  const double* pts;
  float4* out;
  int n;
  double c[3];
  uint32_t* zero;  // optional [n]: K1 row counters (accumulated with atomics) cleared on the way
};

__global__ void engine_pack_kernel(const PackJob* __restrict__ jobs) {
  const PackJob& j = jobs[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < j.n) {
    // pair-interleaved records: K1 reads its column tiles (and its row points) from them
    il_store(j.out, i, pack_point(j.pts[3 * i] - j.c[0], j.pts[3 * i + 1] - j.c[1], j.pts[3 * i + 2] - j.c[2]));
    if (i == j.n - 1 && (j.n & 1)) il_store(j.out, j.n, make_float4(0.f, 0.f, 0.f, 0.f));  // the odd array's last slot
    if (j.zero) j.zero[i] = 0u;
  }
}

struct ProbLayout {
  int C0, M, Ccap;
  size_t in_dbl;   // offset (doubles) of src0 in the input arena: src0, dst0, ori_src, ori_dst
  bool alias_ori;  // the caller passed the same arrays as ori_src / ori_dst (no pre-filter): uploaded once
  size_t in_int;   // offset (ints): keep_mask0, reduce_map0
  double csrc[3], cdst[3];
  double coord_bound;
  int stride;  // mask row stride in words
};

// ---- device-buffer upload (psulvsb_batch_upload_device) -------------------------------------------------------------
// One problem of the engine's part: the caller's device arrays, where they go in the input arena, and its tiles.
struct UploadJob {
  const double* src;
  const double* dst;
  const double* ori_src;  // unused when alias
  const double* ori_dst;
  const int* keep_mask;
  const int* reduce_map;
  unsigned long long in_dbl, in_int;  // ProbLayout::in_dbl / in_int
  int C, M;
  int alias;
  int tile_first;  // first block of this problem (prefix over the part of max(C, M) / UPLOAD_THREADS tiles)
};
// What the upload learns about one problem on the way.  Every field is zero before the launch (one memset) and only
// grows by exact reductions (max, or, add), so the result does not depend on the order of the atomics.
struct UploadSummary {
  unsigned long long lo[2][3];  // min_key of the per-coordinate minimum of src (0) / dst (1)
  unsigned long long hi[2][3];  // max_key of the maximum
  unsigned int nonfinite;       // some coordinate of src, dst or a non-aliased ori_* is NaN or infinite
  unsigned int zeros;           // keep_mask[j] == 0 count
  unsigned int bad_map;         // some keep_mask[j] == 1 has reduce_map[j] outside [0, C)
  unsigned int pad;
};
constexpr int UPLOAD_THREADS = 256;  // points per tile (256 % 3 == 1: see the kernel)

// order-preserving unsigned images of a double (not NaN): max_key orders like the value, min_key is its complement,
// so the maximum of either key gives the minimum / maximum and a zeroed slot is the identity
__host__ __device__ inline unsigned long long max_key_bits(unsigned long long b) {
  return (b >> 63) ? ~b : b | 0x8000000000000000ull;
}
__host__ __device__ inline unsigned long long key_bits_back(unsigned long long k) {
  return (k >> 63) ? k & 0x7FFFFFFFFFFFFFFFull : ~k;
}

__global__ void __launch_bounds__(UPLOAD_THREADS)
    engine_upload_device_kernel(const UploadJob* __restrict__ jobs, int nb, double* __restrict__ in_dbl,
                                int* __restrict__ in_int, UploadSummary* __restrict__ sum) {
  __shared__ unsigned long long part[12][UPLOAD_THREADS / 32];
  int b = 0;
  for (int hi = nb; hi - b > 1;) {  // the problem whose tiles hold this block
    const int mid = (b + hi) >> 1;
    if (jobs[mid].tile_first <= (int)blockIdx.x) b = mid;
    else hi = mid;
  }
  const UploadJob& J = jobs[b];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const long long p0 = (long long)((int)blockIdx.x - J.tile_first) * UPLOAD_THREADS;  // first point of the tile
  // The tile's 3 x 256 doubles of an array are read at 3 p0 + t + 256 r, r = 0..2: coalesced, and since 256 % 3 == 1
  // thread t meets coordinate (t + r) % 3 in its r-th load, i.e. each coordinate exactly once.
  const int t3 = t % 3;
  const size_t n3 = (size_t)3 * (size_t)J.C;
  double* a = in_dbl + J.in_dbl;
  bool bad = false;
  unsigned long long key[12];  // [min 0 / max 1][side][coordinate]
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const double* x = s ? J.dst : J.src;
    double* out = a + (s ? n3 : 0);
    unsigned long long lo_r[3], hi_r[3];  // by load r
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const size_t i = (size_t)(3 * p0) + (size_t)(t + UPLOAD_THREADS * r);
      lo_r[r] = hi_r[r] = 0ull;
      if (i < n3) {
        const double v = x[i];
        out[i] = v;
        bad |= !isfinite(v);
        const unsigned long long k = max_key_bits((unsigned long long)__double_as_longlong(v));
        lo_r[r] = ~k;
        hi_r[r] = k;
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {  // coordinate c came with load (c - t) mod 3
      const int r = (c - t3 + 3) % 3;
      key[3 * s + c] = r == 0 ? lo_r[0] : (r == 1 ? lo_r[1] : lo_r[2]);
      key[6 + 3 * s + c] = r == 0 ? hi_r[0] : (r == 1 ? hi_r[1] : hi_r[2]);
    }
  }
  if (!J.alias) {
    const size_t m3 = (size_t)3 * (size_t)J.M;
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const double* x = s ? J.ori_dst : J.ori_src;
      double* out = a + 2 * n3 + (s ? m3 : 0);
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const size_t i = (size_t)(3 * p0) + (size_t)(t + UPLOAD_THREADS * r);
        if (i < m3) {
          const double v = x[i];
          out[i] = v;
          bad |= !isfinite(v);
        }
      }
    }
  }
  bool zero = false, bad_map = false;
  {
    const long long j = p0 + t;
    if (j < J.M) {
      const int k = J.keep_mask[j], m = J.reduce_map[j];
      int* o = in_int + J.in_int;
      o[j] = k;
      o[J.M + j] = m;
      zero = (k == 0);
      // a kept correspondence's reduced column becomes a line-vector endpoint: it must name a column of src / dst
      bad_map = (k == 1 && (m < 0 || m >= J.C));
    }
  }
#pragma unroll
  for (int q = 0; q < 12; ++q) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) key[q] = max(key[q], __shfl_xor_sync(0xffffffffu, key[q], o));
    if (lane == 0) part[q][wid] = key[q];
  }
  const int any_bad = __syncthreads_or(bad);
  const int n_zero = __syncthreads_count(zero);
  const int any_bad_map = __syncthreads_or(bad_map);
  UploadSummary& S = sum[b];
  if (t < 12) {
    unsigned long long m = 0ull;
    for (int w = 0; w < UPLOAD_THREADS / 32; ++w) m = max(m, part[t][w]);
    if (m) atomicMax(t < 6 ? &S.lo[t / 3][t % 3] : &S.hi[(t - 6) / 3][t % 3], m);
  } else if (t == 32) {
    if (any_bad) atomicOr(&S.nonfinite, 1u);
    if (n_zero) atomicAdd(&S.zeros, (unsigned int)n_zero);
    if (any_bad_map) atomicOr(&S.bad_map, 1u);
  }
}

}  // namespace

class Engine {
 public:
  int device = 0;
  cudaStream_t st = nullptr;
  cudaEvent_t ev_begin = nullptr, ev_end = nullptr, ev_k1 = nullptr, ev_loop = nullptr, ev_m0 = nullptr, ev_m1 = nullptr;
  cudaEvent_t ev_g0 = nullptr, ev_g1 = nullptr;  // around the GNC-TLS launch of a tick
  int B = 0;
  std::vector<ProbLayout> lay;
  std::vector<unsigned long long> reserve;  // self-update edge head-room per job
  size_t in_dbl_total = 0, in_int_total = 0;
  DevBuf d_in_dbl, d_in_int, d_work, d_mask, d_edge, d_jobs, d_misc, d_hist;
  DevBuf d_upload;  // problem table and summaries of upload_device
  unsigned long long sampler_scratch_sig = 0;  // arena layout of the sampler scratch at the last solve
  bool sampler_scratch_clean = false;          // ... and whether that solve ran to completion
  PinBuf h_stage, h_small;
  long long launches = 0;
  double last_ms = 0.0;
  double stage_ms[5] = {0, 0, 0, 0, 0};
  int last_ticks = 0;
  // set by the pool: an event recorded when the pool call began.  The solve then leaves the offsets (ms) of its own
  // begin / end, of the consistency-mask launch and of every GNC-TLS launch relative to it, so that the pool can report
  // device time and per-kernel busy time over several engines running concurrently on their own streams.
  cudaEvent_t origin = nullptr;
  float off_begin = 0.f, off_end = 0.f, off_m0 = 0.f, off_m1 = 0.f;
  std::vector<std::pair<float, float>> gnc_iv, k1_iv;
  int max_chunk = 0;            // largest lock-step sub-batch of a resident batch (0: the whole batch at once)
  int sub_b0 = 0, sub_nb = 0;   // the sub-batch solve_once advances
  std::vector<int> part_ticks;  // ticks of every sub-batch of the last solve
  Comm* comm = nullptr;  // set for one solve by pool_solve_sharded: the consistency rows of the single problem are sharded
  int stage_threads_cap = 12;  // host threads of the staging copy (the pool divides the cores among its engines)

  ~Engine() {
    if (st) cudaStreamSynchronize(st);
    d_in_dbl.release();
    d_in_int.release();
    d_work.release();
    d_mask.release();
    d_edge.release();
    d_jobs.release();
    d_misc.release();
    d_hist.release();
    d_upload.release();
    h_stage.release();
    h_small.release();
    if (ev_begin) cudaEventDestroy(ev_begin);
    if (ev_end) cudaEventDestroy(ev_end);
    if (ev_k1) cudaEventDestroy(ev_k1);
    if (ev_loop) cudaEventDestroy(ev_loop);
    if (ev_m0) cudaEventDestroy(ev_m0);
    if (ev_m1) cudaEventDestroy(ev_m1);
    if (ev_g0) cudaEventDestroy(ev_g0);
    if (ev_g1) cudaEventDestroy(ev_g1);
    if (st) cudaStreamDestroy(st);
  }

  int init(int dev) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return fail(PSULVSB_ERR_NO_DEVICE, "no CUDA device");
    if (dev < 0 || dev >= n) return fail(PSULVSB_ERR_INVALID, "device index out of range");
    cudaDeviceProp prop;
    PSU_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10)
      return fail(PSULVSB_ERR_NO_DEVICE, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                             ", this library is built for sm_100a only");
    device = dev;
    PSU_CUDA(cudaSetDevice(dev));
    PSU_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    PSU_CUDA(cudaEventCreate(&ev_begin));
    PSU_CUDA(cudaEventCreate(&ev_end));
    PSU_CUDA(cudaEventCreate(&ev_k1));
    PSU_CUDA(cudaEventCreate(&ev_loop));
    PSU_CUDA(cudaEventCreate(&ev_m0));
    PSU_CUDA(cudaEventCreate(&ev_m1));
    PSU_CUDA(cudaEventCreate(&ev_g0));
    PSU_CUDA(cudaEventCreate(&ev_g1));
    return PSULVSB_OK;
  }

  int upload(const psulvsb_problem_t* problems, int nb);
  // Device-buffer upload in two halves, so that the pool can have every engine's copy in flight at once: `begin`
  // queues the copy and reductions behind `ready` (an event on the caller's stream), `finish` waits for them and
  // completes the layouts.  The arrays must have passed check_problem and check_device_pointers; `first` is the
  // index of problems[0] in the caller's batch (error messages name problems by that index).
  int upload_device_begin(const psulvsb_problem_t* problems, int nb, cudaEvent_t ready);
  int upload_device_finish(int first);
  int solve(const psulvsb_params_t* params, const uint64_t* seeds, psulvsb_solution_t* solutions,
            psulvsb_trace_t* trace_first);

 private:
  int plan_layout(const psulvsb_problem_t* problems, int nb);
  void make_resident(int nb);
  int solve_once(const psulvsb_params_t* params, const uint64_t* seeds, psulvsb_solution_t* solutions,
                 psulvsb_trace_t* trace_first);
};

namespace {
// Staging copy of one 3 x C point array fused with its bounding box and finiteness check: the source is read once,
// the pinned destination is written with streaming stores (no read-for-ownership traffic on the host memory bus the
// H2D copies of the previous group are reading from at the same time).  lo6 / hi6: per-lane extrema of the period-6
// pattern (x y z x y z), poison: sum of v * 0 (NaN iff some v is NaN or infinite).  dst must be 16-byte aligned.
inline void stage_points(double* dst, const double* src, size_t n_doubles, double lo6[6], double hi6[6], double& poison) {
  for (int k = 0; k < 6; ++k) lo6[k] = hi6[k] = src[k % 3];
  size_t i = 0;
#if defined(__SSE2__)
  if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
    __m128d l0 = _mm_set_pd(src[1], src[0]), l1 = _mm_set_pd(src[0], src[2]), l2 = _mm_set_pd(src[2], src[1]);
    __m128d h0 = l0, h1 = l1, h2 = l2;
    __m128d p0 = _mm_setzero_pd(), p1 = p0, p2 = p0;
    const __m128d zero = _mm_setzero_pd();
    for (; i + 6 <= n_doubles; i += 6) {
      const __m128d a = _mm_loadu_pd(src + i), b = _mm_loadu_pd(src + i + 2), c = _mm_loadu_pd(src + i + 4);
      _mm_stream_pd(dst + i, a);
      _mm_stream_pd(dst + i + 2, b);
      _mm_stream_pd(dst + i + 4, c);
      l0 = _mm_min_pd(l0, a); h0 = _mm_max_pd(h0, a); p0 = _mm_add_pd(p0, _mm_mul_pd(a, zero));
      l1 = _mm_min_pd(l1, b); h1 = _mm_max_pd(h1, b); p1 = _mm_add_pd(p1, _mm_mul_pd(b, zero));
      l2 = _mm_min_pd(l2, c); h2 = _mm_max_pd(h2, c); p2 = _mm_add_pd(p2, _mm_mul_pd(c, zero));
    }
    _mm_sfence();
    double t[2];
    _mm_storeu_pd(t, l0); lo6[0] = t[0]; lo6[1] = t[1];
    _mm_storeu_pd(t, l1); lo6[2] = t[0]; lo6[3] = t[1];
    _mm_storeu_pd(t, l2); lo6[4] = t[0]; lo6[5] = t[1];
    _mm_storeu_pd(t, h0); hi6[0] = t[0]; hi6[1] = t[1];
    _mm_storeu_pd(t, h1); hi6[2] = t[0]; hi6[3] = t[1];
    _mm_storeu_pd(t, h2); hi6[4] = t[0]; hi6[5] = t[1];
    _mm_storeu_pd(t, _mm_add_pd(p0, _mm_add_pd(p1, p2)));
    poison += t[0] + t[1];
  }
#endif
  for (; i < n_doubles; ++i) {  // tail (and the whole array without SSE2)
    const double v = src[i];
    dst[i] = v;
    const int k = (int)(i % 6);
    lo6[k] = v < lo6[k] ? v : lo6[k];
    hi6[k] = v > hi6[k] ? v : hi6[k];
    poison += v * 0.0;
  }
}

// The argument check of both uploads; the message names the problem by b.
int check_problem(const psulvsb_problem_t& p, int b) {
  if (!p.src || !p.dst || !p.ori_src || !p.ori_dst || !p.keep_mask || !p.reduce_map || p.C < 2 || p.M < 1)
    return fail(PSULVSB_ERR_INVALID, "upload: problem " + std::to_string(b) + " has a null array, C < 2 or M < 1");
  return PSULVSB_OK;
}

// The last step of both uploads: the keep_mask zeros give the working-set capacity, the per-side extrema (lo[s] / hi[s]:
// per-coordinate minimum / maximum of src (s = 0) and dst (s = 1)) the centres and the coordinate bound of the FP32
// tiles.  False: a centre or the bound is not finite.
bool finish_layout(ProbLayout& L, int zeros, const double lo[2][3], const double hi[2][3]) {
  L.Ccap = L.C0 + zeros;  // every original correspondence can be appended at most once (registration.cc:828)
  // (differences are translation invariant: each cloud is centred on its own bounding box)
  for (int s = 0; s < 2; ++s) {
    double* c = s ? L.cdst : L.csrc;
    double bound = 0.0;
    for (int r = 0; r < 3; ++r) {
      c[r] = 0.5 * (lo[s][r] + hi[s][r]);
      const double h = 0.5 * (hi[s][r] - lo[s][r]);
      bound = h > bound ? h : bound;
    }
    if (s == 0)
      L.coord_bound = bound;
    else
      L.coord_bound = bound > L.coord_bound ? bound : L.coord_bound;
  }
  L.coord_bound = L.coord_bound * (1.0 + 1e-6) + 1e-30;
  for (int r = 0; r < 3; ++r)
    if (!std::isfinite(L.csrc[r]) || !std::isfinite(L.cdst[r]) || !std::isfinite(L.coord_bound)) return false;
  return true;
}

// the data refusals of both uploads
int refuse_non_finite(int b) {
  return fail(PSULVSB_ERR_INVALID, "upload: problem " + std::to_string(b) + " has non-finite coordinates");
}
int refuse_bad_map(int b) {
  return fail(PSULVSB_ERR_INVALID,
              "upload: problem " + std::to_string(b) + " has keep_mask[j] == 1 with reduce_map[j] outside [0, C)");
}
}  // namespace

// Offsets of every problem in the input arenas, mask strides and aliasing (both uploads).
int Engine::plan_layout(const psulvsb_problem_t* problems, int nb) {
  lay.assign((size_t)nb, ProbLayout());
  size_t od = 0, oi = 0;
  for (int b = 0; b < nb; ++b) {
    const psulvsb_problem_t& p = problems[b];
    if (int rc = check_problem(p, b)) return rc;
    ProbLayout& L = lay[(size_t)b];
    L.C0 = p.C;
    L.M = p.M;
    L.Ccap = p.C;  // + the keep_mask zeros (finish_layout)
    L.stride = (int)align_up((size_t)(p.C + 31) / 32, 8);  // whole 32-byte sectors per row and column tile (K1 stores them as such)
    od = align_up(od, 16);
    L.in_dbl = od;
    L.alias_ori = (p.ori_src == p.src && p.ori_dst == p.dst && p.M == p.C);
    od += (size_t)6 * p.C + (L.alias_ori ? 0 : (size_t)6 * p.M);
    oi = align_up(oi, 32);
    L.in_int = oi;
    oi += (size_t)2 * p.M;
  }
  in_dbl_total = od;
  in_int_total = oi;
  return PSULVSB_OK;
}

void Engine::make_resident(int nb) {
  B = nb;
  reserve.assign((size_t)nb, 0ull);
  for (int b = 0; b < nb; ++b) {
    const ProbLayout& L = lay[(size_t)b];
    if (L.Ccap > L.C0) reserve[(size_t)b] = 65536ull;
  }
}

int Engine::upload(const psulvsb_problem_t* problems, int nb) {
  if (!problems || nb <= 0) return fail(PSULVSB_ERR_INVALID, "upload: no problems");
  if (st) cudaStreamSynchronize(st);  // earlier copies out of the staging buffer (and solves on its contents) are done
  // nothing is resident until this upload has fully succeeded (a failed re-upload must not leave the previous batch
  // size paired with a half-overwritten layout / input arena)
  B = 0;
  reserve.clear();
  PSU_CUDA(cudaSetDevice(device));
  if (int rc = plan_layout(problems, nb)) return rc;
  const size_t od = in_dbl_total, oi = in_int_total;
  const size_t bytes_d = od * sizeof(double), bytes_i = oi * sizeof(int);
  if (int rc = h_stage.ensure(align_up(bytes_d, 256) + bytes_i)) return rc;
  if (int rc = d_in_dbl.ensure(bytes_d)) return rc;
  if (int rc = d_in_int.ensure(bytes_i)) return rc;
  double* hd = reinterpret_cast<double*>(h_stage.p);
  int* hi = reinterpret_cast<int*>(reinterpret_cast<char*>(h_stage.p) + align_up(bytes_d, 256));
  // staging copy + centres / coordinate bound of the FP32 tiles, split over a few host threads (33 MB for a
  // batch of 64 cfg-A pairs: a single-threaded memcpy would cost more than the H2D copy that follows)
  std::atomic<int> bad_problem(-1), bad_map(-1), copy_error(0);
  // a staged group of problems goes to the device at once (its H2D copy overlaps the staging of the next group)
  auto push_group = [&](int g0, int g1) {
    const size_t d0 = lay[(size_t)g0].in_dbl, d1 = (g1 < nb) ? lay[(size_t)g1].in_dbl : od;
    const size_t i0 = lay[(size_t)g0].in_int, i1 = (g1 < nb) ? lay[(size_t)g1].in_int : oi;
    if (cudaMemcpyAsync(reinterpret_cast<double*>(d_in_dbl.p) + d0, hd + d0, (d1 - d0) * sizeof(double),
                        cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(reinterpret_cast<int*>(d_in_int.p) + i0, hi + i0, (i1 - i0) * sizeof(int), cudaMemcpyHostToDevice,
                        st) != cudaSuccess)
      copy_error.store(1);
  };
  auto stage_range = [&](int b0, int b1) {
    if (cudaSetDevice(device) != cudaSuccess) copy_error.store(1);
    int group_begin = b0;
    for (int b = b0; b < b1; ++b) {
      const psulvsb_problem_t& p = problems[b];
      ProbLayout& L = lay[(size_t)b];
      double* d = hd + L.in_dbl;
      if (!L.alias_ori) {
        std::memcpy(d + 6 * (size_t)p.C, p.ori_src, sizeof(double) * 3 * (size_t)p.M);
        std::memcpy(d + 6 * (size_t)p.C + 3 * (size_t)p.M, p.ori_dst, sizeof(double) * 3 * (size_t)p.M);
      }
      std::memcpy(hi + L.in_int, p.keep_mask, sizeof(int) * (size_t)p.M);
      std::memcpy(hi + L.in_int + p.M, p.reduce_map, sizeof(int) * (size_t)p.M);
      int zeros = 0;
      for (int j = 0; j < p.M; ++j) {
        zeros += (p.keep_mask[j] == 0) ? 1 : 0;
        // a kept correspondence's reduced column becomes a line-vector endpoint on the device (inlier_map,
        // registration.cc:1432-1434): it must name a column of src / dst
        if (p.keep_mask[j] == 1 && (p.reduce_map[j] < 0 || p.reduce_map[j] >= p.C)) bad_map.store(b);
      }
      double lo[2][3], hi3[2][3];
      for (int s = 0; s < 2; ++s) {
        const double* pts = s ? p.dst : p.src;
        double lo6[6], hi6[6], poison = 0.0;
        stage_points(d + (s ? 3 * (size_t)p.C : 0), pts, (size_t)3 * p.C, lo6, hi6, poison);
        for (int r = 0; r < 3; ++r) {
          lo[s][r] = lo6[r] < lo6[r + 3] ? lo6[r] : lo6[r + 3];
          hi3[s][r] = hi6[r] > hi6[r + 3] ? hi6[r] : hi6[r + 3];
        }
        if (!L.alias_ori) {
          const double* ori = s ? p.ori_dst : p.ori_src;
          double p6[6] = {0, 0, 0, 0, 0, 0};
          const size_t n_ori = (size_t)3 * p.M;
          for (size_t i = 0; i + 6 <= n_ori; i += 6)
            for (int k = 0; k < 6; ++k) p6[k] += ori[i + k] * 0.0;
          for (size_t i = n_ori - n_ori % 6; i < n_ori; ++i) p6[0] += ori[i] * 0.0;
          poison += p6[0] + p6[1] + p6[2] + p6[3] + p6[4] + p6[5];
        }
        const bool finite = (poison == 0.0);
        if (!finite) bad_problem.store(b);
      }
      if (!finish_layout(L, zeros, lo, hi3)) bad_problem.store(b);
      if (b + 1 - group_begin >= 8 || b + 1 == b1) {  // (measured: groups of 2 finish 0.6 ms later, 13 the same)
        push_group(group_begin, b + 1);
        group_begin = b + 1;
      }
    }
  };
  {
    int nthreads = (int)std::thread::hardware_concurrency();
    if (nthreads > stage_threads_cap) nthreads = stage_threads_cap;
    if (nthreads > nb) nthreads = nb;
    if (nthreads < 1 || bytes_d < (4u << 20)) nthreads = 1;
    if (nthreads == 1) {
      stage_range(0, nb);
    } else {
      std::vector<std::thread> pool;
      for (int t = 0; t < nthreads; ++t)
        pool.emplace_back(stage_range, (int)((long long)nb * t / nthreads), (int)((long long)nb * (t + 1) / nthreads));
      for (auto& th : pool) th.join();
    }
  }
  // The tail of the H2D copies is NOT waited for: everything that consumes the inputs is launched on the same stream,
  // and the host-side set-up of the solve overlaps it.  (The staging buffer is reused by the next upload only, which
  // begins with a stream synchronisation.)
  if (bad_problem.load() >= 0) {
    cudaStreamSynchronize(st);
    return refuse_non_finite(bad_problem.load());
  }
  if (bad_map.load() >= 0) {
    cudaStreamSynchronize(st);
    return refuse_bad_map(bad_map.load());
  }
  if (copy_error.load()) {
    cudaStreamSynchronize(st);
    return fail(PSULVSB_ERR_CUDA, "upload: host-to-device copy failed");
  }
  make_resident(nb);
  return PSULVSB_OK;
}

int Engine::upload_device_begin(const psulvsb_problem_t* problems, int nb, cudaEvent_t ready) {
  if (st) cudaStreamSynchronize(st);  // (as upload: the solves on the previous inputs are done)
  B = 0;
  reserve.clear();
  PSU_CUDA(cudaSetDevice(device));
  if (int rc = plan_layout(problems, nb)) return rc;
  if (int rc = d_in_dbl.ensure(in_dbl_total * sizeof(double))) return rc;
  if (int rc = d_in_int.ensure(in_int_total * sizeof(int))) return rc;
  const size_t table = align_up(sizeof(UploadJob) * (size_t)nb, 256), bytes = table + sizeof(UploadSummary) * (size_t)nb;
  if (int rc = h_small.ensure(bytes)) return rc;
  if (int rc = d_upload.ensure(bytes)) return rc;
  UploadJob* jobs = reinterpret_cast<UploadJob*>(h_small.p);
  long long tiles = 0;
  for (int b = 0; b < nb; ++b) {
    const psulvsb_problem_t& p = problems[b];
    const ProbLayout& L = lay[(size_t)b];
    UploadJob& J = jobs[b];
    J.src = p.src;
    J.dst = p.dst;
    J.ori_src = p.ori_src;
    J.ori_dst = p.ori_dst;
    J.keep_mask = p.keep_mask;
    J.reduce_map = p.reduce_map;
    J.in_dbl = L.in_dbl;
    J.in_int = L.in_int;
    J.C = p.C;
    J.M = p.M;
    J.alias = L.alias_ori ? 1 : 0;
    J.tile_first = (int)tiles;
    tiles += ((long long)(p.C > p.M ? p.C : p.M) + UPLOAD_THREADS - 1) / UPLOAD_THREADS;
  }
  if (tiles > 0x7FFFFFFFll) return fail(PSULVSB_ERR_UNSUPPORTED, "upload_device: more than 2^31 - 1 tiles of 256 points");
  char* d = reinterpret_cast<char*>(d_upload.p);
  PSU_CUDA(cudaStreamWaitEvent(st, ready, 0));  // the caller's work on its inputs comes first
  PSU_CUDA(cudaMemcpyAsync(d, jobs, sizeof(UploadJob) * (size_t)nb, cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaMemsetAsync(d + table, 0, sizeof(UploadSummary) * (size_t)nb, st));
  engine_upload_device_kernel<<<(unsigned)tiles, UPLOAD_THREADS, 0, st>>>(
      reinterpret_cast<const UploadJob*>(d), nb, reinterpret_cast<double*>(d_in_dbl.p),
      reinterpret_cast<int*>(d_in_int.p), reinterpret_cast<UploadSummary*>(d + table));
  ++launches;
  PSU_CUDA(cudaGetLastError());
  PSU_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(h_small.p) + table, d + table, sizeof(UploadSummary) * (size_t)nb,
                           cudaMemcpyDeviceToHost, st));
  return PSULVSB_OK;
}

int Engine::upload_device_finish(int first) {
  PSU_CUDA(cudaStreamSynchronize(st));
  const int nb = (int)lay.size();
  const UploadSummary* sum = reinterpret_cast<const UploadSummary*>(
      reinterpret_cast<const char*>(h_small.p) + align_up(sizeof(UploadJob) * (size_t)nb, 256));
  auto value = [](unsigned long long key) {
    const unsigned long long bits = key_bits_back(key);
    double v;
    std::memcpy(&v, &bits, sizeof(v));
    return v;
  };
  for (int b = 0; b < nb; ++b) {
    double lo[2][3], hi[2][3];
    for (int s = 0; s < 2; ++s)
      for (int r = 0; r < 3; ++r) {
        lo[s][r] = value(~sum[b].lo[s][r]);
        hi[s][r] = value(sum[b].hi[s][r]);
      }
    // (the host path's order: non-finite data or centres first, then the reduce_map check)
    if (sum[b].nonfinite || !finish_layout(lay[(size_t)b], (int)sum[b].zeros, lo, hi)) return refuse_non_finite(first + b);
  }
  for (int b = 0; b < nb; ++b)
    if (sum[b].bad_map) return refuse_bad_map(first + b);
  make_resident(nb);
  return PSULVSB_OK;
}

int Engine::solve(const psulvsb_params_t* params, const uint64_t* seeds, psulvsb_solution_t* solutions,
                  psulvsb_trace_t* trace_first) {
  if (B <= 0) return fail(PSULVSB_ERR_INVALID, "solve: nothing uploaded");
  if (!params || !solutions) return fail(PSULVSB_ERR_INVALID, "solve: null params / solutions");
  if (params->host_round_limit < 0 || params->rotation_max_iterations < 0 || params->inloop_max_iterations < 0)
    return fail(PSULVSB_ERR_INVALID, "solve: negative iteration limits");
  if (params->inlier_selection_mode < 0 || params->inlier_selection_mode > 3)
    return fail(PSULVSB_ERR_INVALID, "solve: inlier_selection_mode must be 0 (PMC_EXACT) .. 3 (NONE)");
  // KCORE_HEU (graph.cc:63-80) returns the maximum k-core when it is larger than threshold * |V| and otherwise the
  // heuristic clique; only the second half exists here (threshold == 1 short-circuits to it in the reference too)
  if (params->inlier_selection_mode == 2 && params->kcore_heuristic_threshold != 1.0)
    return fail(PSULVSB_ERR_UNSUPPORTED,
                "solve: INLIER_SELECTION_MODE::KCORE_HEU with kcore_heuristic_threshold != 1 is not implemented "
                "(PMC_EXACT, PMC_HEU and NONE are)");
  // The resident batch advances in lock-step sub-batches of at most max_chunk registrations (the working arenas are
  // sized per sub-batch, the inputs stay resident); statistics accumulate over them.
  const int step = (max_chunk > 0 && max_chunk < B) ? max_chunk : B;
  const int parts = (B + step - 1) / step;
  double acc_ms = 0.0, acc_stage[5] = {0, 0, 0, 0, 0};
  int acc_ticks = 0;
  float first_begin = 0.f;
  std::vector<std::pair<float, float>> all_gnc, all_k1;
  part_ticks.clear();
  for (int part = 0; part < parts; ++part) {
    sub_b0 = (int)((long long)B * part / parts);
    sub_nb = (int)((long long)B * (part + 1) / parts) - sub_b0;
    const uint64_t* sd = seeds ? seeds + sub_b0 : nullptr;
    psulvsb_params_t pp = *params;
    pp.seed = params->seed + (uint64_t)sub_b0;  // default seeds follow the index in the resident batch
    psulvsb_solution_t* out = solutions + sub_b0;
    for (int attempt = 0; attempt < 6; ++attempt) {
      if (int rc = solve_once(&pp, sd, out, part == 0 ? trace_first : nullptr)) return rc;
      // self-update outgrew the edge head-room of some job: enlarge and redo (results are
      // deterministic, so the retry reproduces the same run with room to finish)
      bool again = false;
      for (int b = 0; b < sub_nb; ++b)
        if (out[b].status == PSULVSB_ERR_CAPACITY) {
          const ProbLayout& L = lay[(size_t)(sub_b0 + b)];
          const unsigned long long full = (unsigned long long)(L.Ccap - L.C0) * (unsigned long long)L.Ccap;
          if (reserve[(size_t)(sub_b0 + b)] < full) {
            unsigned long long r = reserve[(size_t)(sub_b0 + b)] * 8ull;
            reserve[(size_t)(sub_b0 + b)] = r > full ? full : r;
            again = true;
          }
        }
      if (!again) break;
    }
    acc_ms += last_ms;
    for (int i = 0; i < 5; ++i) acc_stage[i] += stage_ms[i];
    acc_ticks = last_ticks > acc_ticks ? last_ticks : acc_ticks;
    part_ticks.push_back(last_ticks);
    all_gnc.insert(all_gnc.end(), gnc_iv.begin(), gnc_iv.end());
    if (origin && off_m1 > off_m0) all_k1.emplace_back(off_m0, off_m1);
    if (part == 0) first_begin = off_begin;
  }
  sub_b0 = 0;
  sub_nb = B;
  last_ms = acc_ms;
  for (int i = 0; i < 5; ++i) stage_ms[i] = acc_stage[i];
  last_ticks = acc_ticks;
  gnc_iv.swap(all_gnc);
  k1_iv.swap(all_k1);
  off_begin = first_begin;
  return PSULVSB_OK;
}

int Engine::solve_once(const psulvsb_params_t* params, const uint64_t* seeds, psulvsb_solution_t* solutions,
                       psulvsb_trace_t* trace_first) {
  PSU_CUDA(cudaSetDevice(device));
  const auto t_begin = std::chrono::steady_clock::now();
  // this call advances the resident problems [sub_b0, sub_b0 + sub_nb) as one lock-step batch (seeds / solutions are
  // already offset by the caller); `B` below is the size of that sub-batch
  const int b0 = sub_b0, B = sub_nb;
  const int local_cap = 512;
  const int host_cap = params->host_round_limit > 0 ? params->host_round_limit : 1;

  // ---- working arena (everything whose size is known before K1)
  std::vector<JobCtl> jobs((size_t)B);
  std::vector<K1Job> k1((size_t)B);
  std::vector<CompactJob> cj((size_t)B);
  std::vector<PackJob> pj((size_t)2 * B);
  const bool ratio = params->estimate_scaling != 0;  // unknown scale: ratio histogram instead of the bit mask
  const bool sharded = comm != nullptr && comm_world(comm) > 1;
  int row_b = 0, row_e = 0;
  if (sharded) {
    if (B != 1 || ratio)
      return fail(PSULVSB_ERR_UNSUPPORTED, "sharded solve: one known-scale registration at a time (independent "
                                           "registrations shard across ranks with no exchange: psulvsb_solve_batch)");
    if (comm_world(comm) > 64) return fail(PSULVSB_ERR_UNSUPPORTED, "sharded solve: at most 64 ranks");
    triangular_row_range(lay[(size_t)b0].C0, comm_rank(comm), comm_world(comm), &row_b, &row_e);
  }
  std::vector<RatioJob> rj(ratio ? (size_t)B : 0);
  struct Misc {
    RatioJob* rj;
    int* bad;
    double* fscale;
    CliqueJob* cq;
    K1Job* k1;
    CompactJob* cj;
    PackJob* pj;
    JobCtl* jobs;
    SampleJob* sl;
    SampleJob* sb;
    GncJob* gj;
    unsigned long long* n_edges;
    unsigned long long* border;
    unsigned long long* counts_all;  // sharded solve: every rank's edge count
    int* n_done;
    psulvsb_solution_t* sols;
  } m;
  {
    Bump bm;
    for (int pass = 0; pass < 2; ++pass) {
      bm.off = 0;
      m.k1 = bm.take<K1Job>((size_t)B);
      m.cj = bm.take<CompactJob>((size_t)B);
      m.pj = bm.take<PackJob>((size_t)2 * B);
      m.jobs = bm.take<JobCtl>((size_t)B);
      m.sl = bm.take<SampleJob>((size_t)B);
      m.sb = bm.take<SampleJob>((size_t)B);
      m.gj = bm.take<GncJob>((size_t)B);
      m.n_edges = bm.take<unsigned long long>((size_t)B);
      m.border = bm.take<unsigned long long>((size_t)B);
      m.counts_all = bm.take<unsigned long long>(64);
      m.n_done = bm.take<int>(4);
      m.sols = bm.take<psulvsb_solution_t>((size_t)B);
      m.rj = bm.take<RatioJob>((size_t)B);
      m.bad = bm.take<int>((size_t)B);
      m.fscale = bm.take<double>((size_t)B);
      m.cq = bm.take<CliqueJob>((size_t)B);
      if (pass == 0) {
        if (int rc = d_misc.ensure(bm.off)) return rc;
        bm.base = reinterpret_cast<char*>(d_misc.p);
      }
    }
  }
  const double* in_dbl = reinterpret_cast<const double*>(d_in_dbl.p);
  const int* in_int = reinterpret_cast<const int*>(d_in_int.p);
  int maxC = 0, maxM = 0;
  {
    Bump bw, bk;
    for (int pass = 0; pass < 2; ++pass) {
      bw.off = 0;
      bk.off = 0;
      for (int b = 0; b < B; ++b) {
        const ProbLayout& L = lay[(size_t)(b0 + b)];
        JobCtl& J = jobs[(size_t)b];
        std::memset(&J, 0, sizeof(J));
        J.C0 = L.C0;
        J.M = L.M;
        J.Ccap = L.Ccap;
        J.src0 = in_dbl + L.in_dbl;
        J.dst0 = J.src0 + 3 * (size_t)L.C0;
        J.ori_src = L.alias_ori ? J.src0 : J.src0 + 6 * (size_t)L.C0;  // read-only on the device
        J.ori_dst = L.alias_ori ? J.dst0 : J.ori_src + 3 * (size_t)L.M;
        J.keep_mask0 = in_int + L.in_int;
        J.reduce_map0 = J.keep_mask0 + L.M;
        J.src = bw.take<double>((size_t)3 * L.Ccap);
        J.dst = bw.take<double>((size_t)3 * L.Ccap);
        J.pts8 = bw.take<double>((size_t)8 * L.Ccap);
        J.residual_history = bw.take<double>((size_t)L.M);
        J.xs = bw.take<double>((size_t)3 * (L.Ccap + 1));
        J.xs_sorted = bw.take<double>(translation_sort_doubles(L.Ccap));
        J.keep_mask = bw.take<int>((size_t)L.M);
        J.reduce_map = bw.take<int>((size_t)L.M);
        J.inlier_counter = bw.take<int>((size_t)L.M);
        J.new_corr = bw.take<int>((size_t)L.M);
        J.inlier_history = bw.take<int>((size_t)L.M);
        J.final_inliers = bw.take<int>((size_t)L.M);
        J.hs_bits = bw.take<uint32_t>(2 * (((size_t)L.M + 31) / 32) + 2);
        J.inlier_map = bw.take<int>((size_t)L.Ccap);
        J.idx = bw.take<int>((size_t)L.Ccap);
        J.adj_stride = (L.Ccap + 31) / 32;
        // the bit matrix is only touched by the last-resort clique escalation; selection NONE never builds it
        J.adj = params->inlier_selection_mode != 3 ? bw.take<uint32_t>(clique_scratch_words(L.Ccap)) : nullptr;
        J.clique_flags = bw.take<uint8_t>((size_t)L.Ccap);
        J.sampled_flags = bw.take<uint8_t>((size_t)L.Ccap);
        J.rot_flags = bw.take<uint8_t>((size_t)L.Ccap);
        J.local_trace = bw.take<psulvsb_local_trace_t>((size_t)local_cap);
        J.host_trace = bw.take<psulvsb_host_trace_t>((size_t)host_cap);
        J.local_trace_cap = local_cap;
        J.host_trace_cap = host_cap;
        J.estimate_scaling = ratio ? 1 : 0;
        J.seed = seeds ? seeds[b] : params->seed + (uint64_t)b;
        const float a = 1 + (((float)L.C0) / (long)L.M);  // registration.cc:669 (float on purpose)
        J.tau = 2 * params->score_noise_bound * a;
        float4* sf = bw.take<float4>(il_records((size_t)L.C0));
        float4* df = bw.take<float4>(il_records((size_t)L.C0));
        K1Job& K = k1[(size_t)b];
        std::memset(&K, 0, sizeof(K));
        K.src = sf;
        K.dst = df;
        K.src64 = J.src0;
        K.dst64 = J.dst0;
        K.n = L.C0;
        K.row_begin = sharded ? row_b : 0;  // sharded: this rank's block of mask rows (other rows keep count 0)
        K.row_end = sharded ? row_e : L.C0;
        K.c = make_k1_consts(2.0 * params->noise_bound * std::sqrt(params->cbar2), L.coord_bound);
        K.mask = ratio ? nullptr : bk.take<uint32_t>((size_t)L.C0 * L.stride);
        K.stride = L.stride;
        K.row_counts = bk.take<uint32_t>((size_t)L.C0);
        if (ratio) {
          RatioJob& Rj = rj[(size_t)b];
          std::memset(&Rj, 0, sizeof(Rj));
          Rj.src64 = J.src0;
          Rj.dst64 = J.dst0;
          Rj.n = L.C0;
          Rj.pair_bin = bk.take<uint32_t>((size_t)L.C0 * (size_t)(L.C0 - 1) / 2 + 1);
          Rj.row_max = bk.take<double>((size_t)L.C0);
          Rj.bp_idx = bk.take<unsigned long long>(RATIO_MAX_GROWTHS);
          Rj.bp_scale = bk.take<double>(RATIO_MAX_GROWTHS);
          Rj.bp_n = bk.take<unsigned int>(1);
          Rj.final_scale = m.fscale + b;
          Rj.peak = bk.take<unsigned int>(4);
          Rj.class_counts = bk.take<unsigned int>((size_t)3 * L.C0);
          Rj.class_offsets = bk.take<unsigned long long>((size_t)3 * L.C0 + 1);
          Rj.n_edges = m.n_edges + b;
          Rj.bad = m.bad + b;
          Rj.active = 1;
        }
        K.border = m.border + b;
        K.active = 1;
        CompactJob& Cj = cj[(size_t)b];
        std::memset(&Cj, 0, sizeof(Cj));
        Cj.mask = K.mask;
        Cj.n = L.C0;
        Cj.stride = L.stride;
        Cj.row_counts = K.row_counts;
        Cj.offsets = bk.take<unsigned long long>((size_t)L.C0 + 1);
        Cj.n_edges = m.n_edges + b;
        Cj.active = 1;
        PackJob& p0 = pj[(size_t)2 * b];
        PackJob& p1 = pj[(size_t)2 * b + 1];
        p0.pts = J.src0;
        p0.out = sf;
        p0.n = L.C0;
        p0.zero = K.row_counts;
        p1.zero = nullptr;
        p1.pts = J.dst0;
        p1.out = df;
        p1.n = L.C0;
        for (int r = 0; r < 3; ++r) {
          p0.c[r] = L.csrc[r];
          p1.c[r] = L.cdst[r];
        }
        maxC = L.C0 > maxC ? L.C0 : maxC;
        maxM = L.M > maxM ? L.M : maxM;
      }
      if (pass == 0) {
        if (int rc = d_work.ensure(bw.off)) return rc;
        if (int rc = d_mask.ensure(bk.off)) return rc;
        bw.base = reinterpret_cast<char*>(d_work.p);
        bk.base = reinterpret_cast<char*>(d_mask.p);
      }
    }
    PSU_CUDA(cudaEventRecord(ev_begin, st));
  }
  PSU_CUDA(cudaMemsetAsync(m.border, 0, sizeof(unsigned long long) * (size_t)B, st));
  PSU_CUDA(cudaMemsetAsync(m.n_done, 0, sizeof(int) * 4, st));
  PSU_CUDA(cudaMemcpyAsync(m.k1, k1.data(), sizeof(K1Job) * (size_t)B, cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaMemcpyAsync(m.cj, cj.data(), sizeof(CompactJob) * (size_t)B, cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaMemcpyAsync(m.pj, pj.data(), sizeof(PackJob) * (size_t)2 * B, cudaMemcpyHostToDevice, st));

  // ---- stage 1: float4 tiles, bit mask, row scan  (unknown scale: ratio histogram, peak, class scan)
  if (ratio) {
    // phase 0: does the histogram grow (a ratio above MaxScale = 10000)?  The final MaxScales size the histograms.
    if (int rc = ratio_count(st, rj, m.rj, maxC, [&](size_t bytes) -> void* { return d_hist.ensure(bytes) ? nullptr : d_hist.p; },
                             ev_m0, ev_m1))
      return rc;
    launches += 8;
  } else {
    {
      dim3 grid((unsigned)((maxC + 255) / 256), (unsigned)(2 * B));
      engine_pack_kernel<<<grid, 256, 0, st>>>(m.pj);
      PSU_CHECK_LAUNCH("engine_pack_kernel");
      ++launches;
    }
    PSU_CUDA(cudaEventRecord(ev_m0, st));
    if (!sharded || row_e > row_b)
      if (int rc = launch_consistency_mask(st, m.k1, B, maxC, sharded ? row_e - row_b : maxC, true)) return rc;
    PSU_CUDA(cudaEventRecord(ev_m1, st));
    ++launches;
    if (int rc = launch_compact_edges(st, m.cj, B, maxC, true, false, false)) return rc;
    ++launches;
  }
  if (int rc = h_small.ensure((sizeof(unsigned long long) + sizeof(int)) * (size_t)B + 64 + 66 * sizeof(unsigned long long)))
    return rc;
  unsigned long long* h_nedges = reinterpret_cast<unsigned long long*>(h_small.p);
  volatile int* h_done = reinterpret_cast<volatile int*>(reinterpret_cast<char*>(h_small.p) + sizeof(unsigned long long) * (size_t)B);
  unsigned long long* h_counts = reinterpret_cast<unsigned long long*>(
      reinterpret_cast<char*>(h_small.p) + align_up((sizeof(unsigned long long) + sizeof(int)) * (size_t)B + 16, 16));
  std::vector<unsigned long long> shard_off;  // sharded: rank r's edges are [shard_off[r], shard_off[r + 1]) of the list
  if (sharded) {
    // every rank's edge count (8 bytes each) -> the offsets of the rank blocks in the global, row-major edge list
    if (int rc = comm_allgather_u64(comm, st, m.n_edges, m.counts_all)) return rc;
    PSU_CUDA(cudaMemcpyAsync(h_counts, m.counts_all, sizeof(unsigned long long) * (size_t)comm_world(comm),
                             cudaMemcpyDeviceToHost, st));
    PSU_CUDA(cudaStreamSynchronize(st));
    shard_off.assign((size_t)comm_world(comm) + 1, 0ull);
    for (int r = 0; r < comm_world(comm); ++r) shard_off[(size_t)r + 1] = shard_off[(size_t)r] + h_counts[r];
    h_nedges[0] = shard_off.back();
    PSU_CUDA(cudaMemcpyAsync(m.n_edges, h_nedges, sizeof(unsigned long long), cudaMemcpyHostToDevice, st));  // n_red
  } else {
    PSU_CUDA(cudaMemcpyAsync(h_nedges, m.n_edges, sizeof(unsigned long long) * (size_t)B, cudaMemcpyDeviceToHost, st));
    PSU_CUDA(cudaStreamSynchronize(st));
  }

  // ---- edge arena, sized from the measured reduced-set sizes.  The reduced set is EdgeNarrow (4 bytes per edge) when
  // every working set of the chunk fits 16-bit point indices; the sharded exchange moves EdgeWide lists.
  bool narrow = !sharded && !debug_knobs().edge_wide;
  for (int b = 0; b < B; ++b) narrow = narrow && edge_narrow_fits(lay[(size_t)(b0 + b)].Ccap);
  const int grid_ctas_max = sm_count() / (B > 0 ? B : 1);  // CTAs per registration the GNC kernel's grid mode may use
  unsigned long long max_cap = 0, max_nred = 0;
  // every sample of the chunk goes to the sampler's on-chip pass except the (1.0, 1.0) escalation, whose window is
  // longer than the draw cache and the bucket lists cover: neither is ever read, so neither is reserved
  bool sample_onchip = true;
  for (int b = 0; b < B; ++b)
    sample_onchip = sample_onchip && sample_onchip_bound(std::max(h_nedges[b] + reserve[(size_t)(b0 + b)], 64ull));
  {
    Bump be;
    for (int pass = 0; pass < 2; ++pass) {
      be.off = 0;
      for (int b = 0; b < B; ++b) {
        JobCtl& J = jobs[(size_t)b];
        unsigned long long cap = h_nedges[b] + reserve[(size_t)(b0 + b)];
        if (cap < 64) cap = 64;
        J.edge_cap = cap;
        J.edges = narrow ? (void*)be.take<EdgeNarrow::T>((size_t)cap) : (void*)be.take<EdgeWide::T>((size_t)cap);
        // (the (1.0, 1.0) rate pair draws ALL n values by rejection -- a random order, ~n (ln n + 10.6) draws)
        J.first_words = sample_table_words(cap, sample_default_max_draws(cap, cap));
        J.first = be.take<uint32_t>((size_t)J.first_words);
        J.draws_cap = sample_onchip ? 0ull : (cap + 3) & ~3ull;  // covers every rate pair below (1.0, 1.0); longer windows recompute
        J.draws = J.draws_cap ? be.take<uint32_t>((size_t)J.draws_cap) : nullptr;
        J.chunk_prefix = be.take<unsigned long long>((size_t)sample_chunk_slots(sample_default_max_draws(cap, cap)));
        J.ticket = be.take<unsigned int>(4);
        // bucket lists of the sampler: sized for the L sample at the largest rate below 1.0 (0.5 -> ~0.7 cap draws)
        J.blist_cap = sample_onchip ? 0ull : sample_list_entries(cap, cap);
        J.blist = J.blist_cap ? be.take<uint32_t>((size_t)J.blist_cap) : nullptr;
        J.bcount = J.blist ? be.take<unsigned int>((size_t)sample_list_counters()) : nullptr;
        J.vbits = be.take<uint32_t>((size_t)((cap + 31) / 32 + 32));
        J.L_sampled = be.take<uint32_t>((size_t)cap);
        J.basic_idx = be.take<uint32_t>((size_t)cap);
        J.basic_edges = be.take<uint2>((size_t)cap);
        J.weights = be.take<double>((size_t)cap);
        // covers the basic subsets up to the (0.5, 0.3) rate pair; the (1, 1) escalation recomputes the rest
        J.lv_cap = cap / 6 + 64;
        J.lv = be.take<double>((size_t)6 * J.lv_cap);
        J.gnc_perm = be.take<uint32_t>((size_t)2 * J.lv_cap);
        if (grid_ctas_max >= 16) {  // few registrations: the GNC kernel may spread each over many SMs (grid mode)
          J.gnc_grid_red = be.take<double>((size_t)grid_ctas_max * GNC_GRID_RED_DOUBLES);
          J.gnc_grid_bar = be.take<unsigned int>(4);
        }
        J.pruned_edges = ratio ? be.take<uint2>((size_t)cap) : nullptr;
        if (ratio) {
          rj[(size_t)b].edges = J.edges;
          rj[(size_t)b].cap = cap;
        }
        // (sharded: this rank's rows land at their place in the global list)
        cj[(size_t)b].edges = static_cast<EdgeWide::T*>(J.edges) + (sharded && be.base ? shard_off[(size_t)comm_rank(comm)] : 0ull);
        cj[(size_t)b].cap = cap - (sharded ? shard_off[(size_t)comm_rank(comm)] : 0ull);
        max_cap = cap > max_cap ? cap : max_cap;
        max_nred = h_nedges[b] > max_nred ? h_nedges[b] : max_nred;
      }
      if (pass == 0) {
        if (int rc = d_edge.ensure(be.off)) return rc;
        be.base = reinterpret_cast<char*>(d_edge.p);
      }
    }
  }
  if (max_cap >= 0x7FFFFFF0ull) return fail(PSULVSB_ERR_UNSUPPORTED, "reduced set exceeds the 31-bit sample / line-vector indices");
  PSU_CUDA(cudaMemcpyAsync(m.jobs, jobs.data(), sizeof(JobCtl) * (size_t)B, cudaMemcpyHostToDevice, st));
  if (ratio) {
    if (int rc = ratio_emit(st, rj, m.rj, maxC, narrow)) return rc;
  } else {
    PSU_CUDA(cudaMemcpyAsync(m.cj, cj.data(), sizeof(CompactJob) * (size_t)B, cudaMemcpyHostToDevice, st));
    if (int rc = launch_compact_edges(st, m.cj, B, maxC, false, true, narrow)) return rc;
    if (sharded) {  // every rank receives every other rank's block of the edge list (8 bytes per edge, over NVLink)
      std::vector<unsigned long long> off32(shard_off);
      for (auto& o : off32) o *= 2ull;
      if (int rc = comm_allgatherv_inplace_u32(comm, st, reinterpret_cast<uint32_t*>(jobs[0].edges), off32.data())) return rc;
    }
  }
  ++launches;

  EngineParams P;
  P.caller = SubParams{params->noise_bound, params->cbar2, params->rotation_max_iterations, params->rotation_gnc_factor,
                       params->rotation_cost_threshold};
  P.inloop = SubParams{params->inloop_noise_bound, params->inloop_cbar2, params->inloop_max_iterations,
                       params->inloop_gnc_factor, params->inloop_cost_threshold};
  P.pr_noise = 2 * params->score_noise_bound;
  P.score_sigma = params->score_noise_bound;
  P.rotation_similar = params->rotation_similar;
  P.local_max_iter = params->local_max_iter;
  P.tpro_host = params->tpro_host;
  P.tpro_local = params->tpro_local;
  P.host_round_limit = params->host_round_limit;
  P.wallclock_cap_s = params->wallclock_cap_s;
  P.self_update = params->self_update;
  P.inlier_selection_mode = params->inlier_selection_mode;
  P.max_local_iters = 4096;
  // one registration's M points scored by ONE CTA is fine at M = 5000 (and two launches per tick would cost a batch of
  // small problems more than it gains); from 32 768 points on the scoring gets a grid-wide kernel of its own
  P.split_host_scoring = (maxM >= 32768) ? 1 : 0;
  P.sampler_counters = (int)sample_list_counters();
  {
    // The sampler leaves its accept bitmask and value bitmap zeroed after every use.  They are cleared here only when
    // that cannot be relied on: a new arena layout (other pointers / sizes than the last COMPLETED solve) or a
    // previous solve that ended early.  Saves a ~2.5 MB memset per registration and solve.
    unsigned long long sig = 1469598103934665603ull;
    auto mix = [&](unsigned long long v) { sig = (sig ^ v) * 1099511628211ull; };
    for (int b = 0; b < B; ++b) {
      const JobCtl& J = jobs[(size_t)b];
      mix((unsigned long long)(uintptr_t)J.first);
      mix(J.first_words);
      mix((unsigned long long)(uintptr_t)J.vbits);
      mix(J.edge_cap);
    }
    P.zero_sampler_scratch = (sampler_scratch_sig == sig && sampler_scratch_clean) ? 0 : 1;
    sampler_scratch_sig = sig;
    sampler_scratch_clean = false;  // until this solve completes
  }
  {
    // CTAs per job: enough that a lone large registration's copies use the whole GPU, one when the batch fills it
    int init_y = (int)(((long long)sm_count() * 2 + B - 1) / B);
    const int by_size = (std::max(maxM, maxC) + 4 * kCtlThreads - 1) / (4 * kCtlThreads);
    if (init_y > by_size) init_y = by_size;
    if (init_y < 1) init_y = 1;
    engine_init_kernel<<<dim3((unsigned)B, (unsigned)init_y), kCtlThreads, 0, st>>>(m.jobs, m.sl, m.sb, m.gj, m.cq, m.n_edges, P,
                                                                                    m.n_done);
  }
  PSU_CHECK_LAUNCH("engine_init_kernel");
  ++launches;
  PSU_CUDA(cudaEventRecord(ev_k1, st));

  // ---- ticks
  // CTAs per registration follow the registrations still RUNNING (the previous tick's count): the CTAs of finished
  // jobs leave at once, so the last stragglers of a batch get 2 / 4 / 8 SMs each instead of one (the tail ticks of a
  // lock-step batch are what weak scaling loses: the slowest rank of 8 ran 25.5 ms against 20.8 ms on one GPU)
  int n_running = B;
  int max_ccap = 0;
  for (int b = 0; b < B; ++b) max_ccap = lay[(size_t)(b0 + b)].Ccap > max_ccap ? lay[(size_t)(b0 + b)].Ccap : max_ccap;
  const unsigned long long draws_bound = sample_default_max_draws(max_cap, max_cap / 8 + 1);
  int ticks = 0;
  double gnc_ms = 0.0;
  gnc_iv.clear();
  const int max_ticks = P.max_local_iters + P.host_round_limit + 8;
  bool round_start_pending = true;  // every job begins with a round start
  bool clique_pending = false;
  while (true) {
    const double elapsed =
        std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t_begin).count() / 1e6;
    if (round_start_pending) {
      if (int rc = launch_round_start(st, B, m.jobs, m.sl, m.sb, m.gj, m.cq, P, m.n_done, narrow)) return rc;
      if (int rc = launch_sample(st, m.sl, B, draws_bound, max_cap, max_ccap, narrow)) return rc;
      launches += 5;
    }
    if (int rc = launch_sample(st, m.sb, B, draws_bound, max_cap, 0, narrow)) return rc;
    if (ratio) {
      engine_scale_kernel<<<B, kCtlThreads, 0, st>>>(m.jobs, m.gj, m.cq, P);
      PSU_CHECK_LAUNCH("engine_scale_kernel");
      ++launches;
    }
    if (clique_pending) {  // some registration is in its clique round (rare, last escalation)
      int maxCcap = 0;
      for (int b = 0; b < B; ++b) maxCcap = lay[(size_t)(b0 + b)].Ccap > maxCcap ? lay[(size_t)(b0 + b)].Ccap : maxCcap;
      // PMC_EXACT: greedy lower bound + exact improvement search; PMC_HEU / KCORE_HEU: the heuristic clique only
      // (graph.cc:86-121).  max_clique_time_limit has no counterpart: the search has a node budget instead.
      if (int rc = launch_max_clique(st, m.cq, B, maxCcap, (maxCcap + 31) / 32, max_cap, params->inlier_selection_mode == 0))
        return rc;
      launches += 8;
    }
    PSU_CUDA(cudaEventRecord(ev_g0, st));
    int gnc_cluster = gnc_cluster_for(n_running);
    // few registrations with very many line vectors (cfg-B: one with ~ 10^6): grid mode, as many CTAs per registration as
    // give each a few thousand line vectors and as the SMs allow
    if (gnc_cluster == 8 && grid_ctas_max >= 16) {
      const long long k_est = (long long)(0.03 * (double)max_nred);
      const long long g = std::min<long long>(grid_ctas_max, k_est / 4096);
      if (g >= 16) gnc_cluster = (int)g;
    }
    int gnc_cap = (int)((0.03 * (double)max_nred) / (double)gnc_cluster) + 64;
    gnc_cap = (gnc_cap + 31) & ~31;
    if (gnc_cap > gnc_default_capacity()) gnc_cap = gnc_default_capacity();
    if (int rc = launch_gnc_tls(st, m.gj, B, gnc_cap, gnc_cluster, n_running)) return rc;
    PSU_CUDA(cudaEventRecord(ev_g1, st));
    engine_local_control_kernel<<<B, kCtlThreads, 0, st>>>(m.jobs, m.sl, m.sb, m.gj, m.cq, P, elapsed, m.n_done);
    PSU_CHECK_LAUNCH("engine_local_control_kernel");
    launches += 5;
    if (P.split_host_scoring) {  // large M: the host scoring of a tick on the whole GPU (both exit at once when no job asks)
      engine_host_score_kernel<<<dim3((unsigned)((maxM + kCtlThreads - 1) / kCtlThreads), (unsigned)B), kCtlThreads, 0, st>>>(
          m.jobs, P);
      PSU_CHECK_LAUNCH("engine_host_score_kernel");
      engine_host_finish_kernel<<<B, kCtlThreads, 0, st>>>(m.jobs, m.sb, m.gj, m.cq, P, elapsed, m.n_done);
      PSU_CHECK_LAUNCH("engine_host_finish_kernel");
      launches += 2;
    }
    ++ticks;
    PSU_CUDA(cudaMemcpyAsync((void*)h_done, m.n_done, 3 * sizeof(int), cudaMemcpyDeviceToHost, st));
    PSU_CUDA(cudaStreamSynchronize(st));
    {
      float g = 0.f;
      if (cudaEventElapsedTime(&g, ev_g0, ev_g1) == cudaSuccess) gnc_ms += g;  // (the tick's poll already synchronised)
      float a = 0.f;
      if (origin && cudaEventElapsedTime(&a, origin, ev_g0) == cudaSuccess) gnc_iv.emplace_back(a, a + g);
    }
    if (h_done[0] >= B) break;
    n_running = B - h_done[0];
    round_start_pending = h_done[1] > 0;
    clique_pending = h_done[2] > 0 && params->inlier_selection_mode != 3;
    if (ticks >= max_ticks) return fail(PSULVSB_ERR_INTERNAL, "engine did not converge within the tick limit");
  }
  last_ticks = ticks;
  PSU_CUDA(cudaEventRecord(ev_loop, st));
  engine_refine_kernel<<<B, kCtlThreads, 0, st>>>(m.jobs, m.sols, m.border);
  PSU_CHECK_LAUNCH("engine_refine_kernel");
  ++launches;
  PSU_CUDA(cudaMemcpyAsync(solutions, m.sols, sizeof(psulvsb_solution_t) * (size_t)B, cudaMemcpyDeviceToHost, st));
  PSU_CUDA(cudaEventRecord(ev_end, st));
  PSU_CUDA(cudaStreamSynchronize(st));
  sampler_scratch_clean = true;  // every sample of this solve ran all its passes
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ev_begin, ev_end);
  last_ms = ms;
  cudaEventElapsedTime(&ms, ev_begin, ev_k1);
  stage_ms[0] = ms;
  cudaEventElapsedTime(&ms, ev_k1, ev_loop);
  stage_ms[1] = ms;
  cudaEventElapsedTime(&ms, ev_loop, ev_end);
  stage_ms[4] = ms;
  cudaEventElapsedTime(&ms, ev_m0, ev_m1);
  stage_ms[2] = ms;  // the consistency-mask kernel alone (one launch over the whole batch)
  stage_ms[3] = gnc_ms;  // the GNC-TLS launches of all ticks
  if (origin) {
    cudaEventElapsedTime(&off_begin, origin, ev_begin);
    cudaEventElapsedTime(&off_end, origin, ev_end);
    cudaEventElapsedTime(&off_m0, origin, ev_m0);
    cudaEventElapsedTime(&off_m1, origin, ev_m1);
  }

  if (trace_first) {
    JobCtl j0;
    PSU_CUDA(cudaMemcpy(&j0, m.jobs, sizeof(JobCtl), cudaMemcpyDeviceToHost));
    trace_first->local_n = 0;
    trace_first->host_n = 0;
    if (trace_first->local && trace_first->local_cap > 0) {
      const int n = j0.n_local_trace < trace_first->local_cap ? j0.n_local_trace : trace_first->local_cap;
      if (n > 0)
        PSU_CUDA(cudaMemcpy(trace_first->local, j0.local_trace, sizeof(psulvsb_local_trace_t) * (size_t)n,
                            cudaMemcpyDeviceToHost));
      trace_first->local_n = n;
    }
    if (trace_first->host && trace_first->host_cap > 0) {
      const int n = j0.n_host_trace < trace_first->host_cap ? j0.n_host_trace : trace_first->host_cap;
      if (n > 0)
        PSU_CUDA(cudaMemcpy(trace_first->host, j0.host_trace, sizeof(psulvsb_host_trace_t) * (size_t)n,
                            cudaMemcpyDeviceToHost));
      trace_first->host_n = n;
    }
    if (trace_first->final_inliers)
      PSU_CUDA(cudaMemcpy(trace_first->final_inliers, j0.final_inliers, sizeof(int) * (size_t)j0.M, cudaMemcpyDeviceToHost));
    if (trace_first->inlier_counter)
      PSU_CUDA(cudaMemcpy(trace_first->inlier_counter, j0.inlier_counter, sizeof(int) * (size_t)j0.M, cudaMemcpyDeviceToHost));
    if (trace_first->reduce_map_out)
      PSU_CUDA(cudaMemcpy(trace_first->reduce_map_out, j0.reduce_map, sizeof(int) * (size_t)j0.M, cudaMemcpyDeviceToHost));
  }
  return PSULVSB_OK;
}

// ---- engine pool -----------------------------------------------------------------------------
// A handle owns a small pool of engines on one device, each with its own stream and arenas.  A batch larger than one
// lock-step chunk is cut into chunks that advance CONCURRENTLY, one per engine, each driven by its own host thread:
//   * a chunk's latency-bound phases (GNC-TLS, control kernels, the per-tick poll) overlap another chunk's
//     bandwidth-bound ones (sampler passes, compaction), and the straggler ticks at the end of one chunk -- a handful of
//     registrations on a few SMs -- overlap the bulk of the next instead of idling the device;
//   * with host buffers (psulvsb_solve_batch) the chunks are handed out dynamically, so the staging + H2D copy of chunk
//     k + 1 runs while chunk k is being solved.
// Results do not depend on the partition: every registration's state and sample stream are its own.
namespace {
// length of the union of intervals (ms)
double union_ms(std::vector<std::pair<float, float>>& iv) {
  if (iv.empty()) return 0.0;
  std::sort(iv.begin(), iv.end());
  double total = 0.0;
  float lo = iv[0].first, hi = iv[0].second;
  for (size_t i = 1; i < iv.size(); ++i) {
    if (iv[i].first > hi) {
      total += hi - lo;
      lo = iv[i].first;
      hi = iv[i].second;
    } else if (iv[i].second > hi) {
      hi = iv[i].second;
    }
  }
  return total + (hi - lo);
}
}  // namespace

namespace {
int available_cpus() {
  cpu_set_t set;
  CPU_ZERO(&set);
  if (sched_getaffinity(0, sizeof(set), &set) == 0) {
    const int n = CPU_COUNT(&set);
    if (n > 0) return n;
  }
  const int hw = (int)std::thread::hardware_concurrency();
  return hw > 0 ? hw : 1;
}
}  // namespace

class EnginePool {
 public:
  int device = 0;
  int chunk = 0;  // registrations per lock-step chunk (0: one per SM)
  int lanes = 0;  // engines that may run concurrently (0: default)
  int host_threads = 0;  // host threads for staging (0: the CPUs available to the process)
  std::vector<Engine*> eng;
  cudaEvent_t origin = nullptr;
  cudaEvent_t ready = nullptr;  // upload_device: recorded on the caller's stream
  std::vector<int> res_begin;  // resident partition: engine e holds problems [res_begin[e], res_begin[e + 1])
  int resident_B = 0;
  double last_ms = 0.0;
  double stage_ms[5] = {0, 0, 0, 0, 0};
  int last_ticks = 0;
  std::vector<int> chunk_ticks;  // ticks of every chunk of the last call
  long long retired_launches = 0;

  ~EnginePool() {
    stop_workers();
    for (Engine* e : eng) delete e;
    if (origin) cudaEventDestroy(origin);
    if (ready) cudaEventDestroy(ready);
    if (mark_st) cudaStreamDestroy(mark_st);
  }
  int init(int dev) {
    device = dev;
    Engine* e = new Engine();
    if (int rc = e->init(dev)) {
      delete e;
      return rc;
    }
    eng.push_back(e);
    PSU_CUDA(cudaEventCreate(&origin));
    return ensure_engines(1);
  }
  int chunk_size() const { return chunk > 0 ? chunk : 4 * sm_count(); }
  int lane_count() const { return lanes > 0 ? lanes : 2; }
  int ensure_engines(int n) {
    while ((int)eng.size() < n) {
      Engine* e = new Engine();
      if (int rc = e->init(device)) {
        delete e;
        return rc;
      }
      eng.push_back(e);
    }
    // host threads of the staging copies: the CPUs this PROCESS may run on (its affinity mask / cgroup share, not the
    // machine's core count), or the caller's figure (psulvsb_set_host_threads: e.g. cores / ranks on a multi-GPU node,
    // where eight ranks staging with a dozen threads each oversubscribe a 32-CPU container), shared by the engines
    // (uploads take turns -- upload_mu -- so the uploading engine may have them all but one per solving lane)
    int hw = host_threads > 0 ? host_threads : available_cpus();
    int per = hw - (n > 1 ? n - 1 : 0);
    per = per < 1 ? 1 : (per > 12 ? 12 : per);
    for (Engine* e : eng) {
      e->stage_threads_cap = per;
      e->max_chunk = chunk_size();
    }
    return PSULVSB_OK;
  }
  long long launch_count() const {
    long long n = retired_launches;
    for (const Engine* e : eng) n += e->launches;
    return n;
  }

  // statistics of a call from the engines that took part; `records` holds one entry per chunk
  struct ChunkRecord {
    float off_begin, off_end;
    double stage[5];
    int ticks;
    std::vector<int> part_ticks;
    std::vector<std::pair<float, float>> gnc, k1;
  };
  static ChunkRecord record_of(const Engine* e) {
    ChunkRecord r;
    r.off_begin = e->off_begin;
    r.off_end = e->off_end;
    r.k1 = e->k1_iv;
    for (int i = 0; i < 5; ++i) r.stage[i] = e->stage_ms[i];
    r.ticks = e->last_ticks;
    r.part_ticks = e->part_ticks;
    r.gnc = e->gnc_iv;
    return r;
  }
  void fold(std::vector<ChunkRecord>& recs) {
    last_ms = 0.0;
    last_ticks = 0;
    chunk_ticks.clear();
    for (int i = 0; i < 5; ++i) stage_ms[i] = 0.0;
    std::vector<std::pair<float, float>> k1, gnc;
    for (const ChunkRecord& r : recs) {
      last_ms = r.off_end > last_ms ? r.off_end : last_ms;
      last_ticks = r.ticks > last_ticks ? r.ticks : last_ticks;
      chunk_ticks.insert(chunk_ticks.end(), r.part_ticks.begin(), r.part_ticks.end());
      stage_ms[0] += r.stage[0] / (double)recs.size();
      stage_ms[1] += r.stage[1] / (double)recs.size();
      stage_ms[4] += r.stage[4] / (double)recs.size();
      k1.insert(k1.end(), r.k1.begin(), r.k1.end());
      gnc.insert(gnc.end(), r.gnc.begin(), r.gnc.end());
    }
    stage_ms[2] = union_ms(k1);   // time during which a consistency-mask launch of some chunk was running
    stage_ms[3] = union_ms(gnc);  // ... a GNC-TLS launch of some chunk
  }

  // ---- pipelined batches (psulvsb_batch_submit / psulvsb_batch_wait) -------------------------------
  // One persistent host thread per lane, each bound to its own engine, pulls lock-step chunks from a queue that runs
  // ACROSS calls: while one lane solves the last chunk of batch n, the other already stages and copies the first chunk
  // of batch n + 1, so a stream of batches keeps the device busy and the uploads disappear behind the solves.
  struct Call {
    uint64_t id = 0;
    psulvsb_params_t params;
    const psulvsb_problem_t* problems = nullptr;
    int B = 0;
    std::vector<uint64_t> seeds;
    psulvsb_solution_t* solutions = nullptr;
    std::vector<int> begin;
    int n_chunks = 0, next_chunk = 0, done_chunks = 0;
    int rc = PSULVSB_OK;
    std::string msg;
    std::vector<ChunkRecord> recs;
    cudaEvent_t origin = nullptr;
  };
  std::mutex upload_mu;
  std::mutex q_mu;
  std::condition_variable q_work, q_done, q_solve;
  int solving = 0;  // chunks being solved right now
  std::deque<std::shared_ptr<Call>> q_pending;          // calls with chunks still to hand out, in submission order
  std::map<uint64_t, std::shared_ptr<Call>> q_calls;    // submitted and not yet waited for
  std::vector<std::thread> workers;
  bool q_stop = false;
  uint64_t next_ticket = 1;
  int in_flight = 0;  // calls submitted and not yet complete
  cudaStream_t mark_st = nullptr;

  void worker_main(int w) {
    cudaSetDevice(device);
    Engine* e = eng[(size_t)w];
    for (;;) {
      std::shared_ptr<Call> call;
      int c = -1;
      {
        std::unique_lock<std::mutex> lk(q_mu);
        q_work.wait(lk, [&] { return q_stop || !q_pending.empty(); });
        if (q_stop) return;
        call = q_pending.front();
        c = call->next_chunk++;
        if (call->next_chunk >= call->n_chunks) q_pending.pop_front();
      }
      int rc = PSULVSB_OK;
      std::string msg;
      bool skip;
      {
        std::lock_guard<std::mutex> lk(q_mu);
        skip = call->rc != PSULVSB_OK;  // an earlier chunk of the call failed: its result is void anyway
      }
      if (!skip) {
        const int b0 = call->begin[(size_t)c], nb = call->begin[(size_t)c + 1] - b0;
        e->origin = call->origin;
        {
          // one upload at a time: it has all the staging threads and the whole PCIe link
          std::lock_guard<std::mutex> up(upload_mu);
          rc = e->upload(call->problems + b0, nb);
          if (!rc && cudaStreamSynchronize(e->st) != cudaSuccess)  // (the copies too: the link is the next upload's now)
            rc = fail(PSULVSB_ERR_CUDA, "upload: copy failed");
        }
        if (!rc) {
          // at most lane_count() chunks are being solved at a time; the extra worker has the next chunk uploaded by
          // the time one of them finishes (chunks that run together finish together, whatever their head start, so
          // without it every lane would upload while the device idles)
          {
            std::unique_lock<std::mutex> lk(q_mu);
            q_solve.wait(lk, [&] { return solving < lane_count(); });
            ++solving;
          }
          rc = e->solve(&call->params, call->seeds.data() + b0, call->solutions + b0, nullptr);
          {
            std::lock_guard<std::mutex> lk(q_mu);
            --solving;
          }
          q_solve.notify_one();
        }
        if (rc) msg = psulvsb_last_error();
        else call->recs[(size_t)c] = record_of(e);
      }
      {
        std::lock_guard<std::mutex> lk(q_mu);
        if (rc && call->rc == PSULVSB_OK) {
          call->rc = rc;
          call->msg = msg;
        }
        if (++call->done_chunks == call->n_chunks) {
          --in_flight;
          q_done.notify_all();
        }
      }
    }
  }
  int start_workers() {
    const int n = lane_count() + 1;  // one more than may solve at a time: it uploads meanwhile
    if ((int)workers.size() == n) return PSULVSB_OK;
    stop_workers();
    if (int rc = ensure_engines(n)) return rc;
    if (!mark_st) PSU_CUDA(cudaStreamCreateWithFlags(&mark_st, cudaStreamNonBlocking));
    q_stop = false;
    for (int w = 0; w < n; ++w) workers.emplace_back([this, w] { worker_main(w); });
    return PSULVSB_OK;
  }
  void stop_workers() {
    {
      std::lock_guard<std::mutex> lk(q_mu);
      q_stop = true;
    }
    q_work.notify_all();
    for (auto& t : workers) t.join();
    workers.clear();
  }
  // every other entry point runs on the caller's thread with the engines to itself
  void drain() {
    std::unique_lock<std::mutex> lk(q_mu);
    q_done.wait(lk, [&] { return in_flight == 0; });
  }
  int submit(const psulvsb_params_t* params, const psulvsb_problem_t* problems, int B, const uint64_t* seeds,
             psulvsb_solution_t* solutions, uint64_t* ticket) {
    if (!params || !problems || !solutions || !ticket || B <= 0)
      return fail(PSULVSB_ERR_INVALID, "batch_submit: NULL argument or B <= 0");
    PSU_CUDA(cudaSetDevice(device));
    if (int rc = start_workers()) return rc;
    auto call = std::make_shared<Call>();
    call->params = *params;
    call->problems = problems;
    call->B = B;
    call->solutions = solutions;
    call->seeds.resize((size_t)B);
    for (int b = 0; b < B; ++b) call->seeds[(size_t)b] = seeds ? seeds[b] : params->seed + (uint64_t)b;
    const int ch = chunk_size();
    call->n_chunks = (B + ch - 1) / ch;
    partition(B, call->n_chunks, call->begin);
    call->recs.resize((size_t)call->n_chunks);
    PSU_CUDA(cudaEventCreate(&call->origin));
    PSU_CUDA(cudaEventRecord(call->origin, mark_st));
    {
      std::lock_guard<std::mutex> lk(q_mu);
      resident_B = 0;
      call->id = next_ticket++;
      q_calls[call->id] = call;
      q_pending.push_back(call);
      ++in_flight;
    }
    q_work.notify_all();
    *ticket = call->id;
    return PSULVSB_OK;
  }
  int wait(uint64_t ticket) {
    std::shared_ptr<Call> call;
    {
      std::unique_lock<std::mutex> lk(q_mu);
      auto it = q_calls.find(ticket);
      if (it == q_calls.end()) return fail(PSULVSB_ERR_INVALID, "batch_wait: unknown ticket");
      call = it->second;
      q_done.wait(lk, [&] { return call->done_chunks == call->n_chunks; });
      q_calls.erase(it);
    }
    cudaEventDestroy(call->origin);
    if (call->rc) return fail(call->rc, call->msg);
    fold(call->recs);
    return PSULVSB_OK;
  }

  int solve_one(const psulvsb_params_t* params, const psulvsb_problem_t* problem, psulvsb_solution_t* solution,
                psulvsb_trace_t* trace) {
    drain();
    resident_B = 0;
    Engine* e = eng[0];
    PSU_CUDA(cudaSetDevice(device));
    PSU_CUDA(cudaEventRecord(origin, e->st));
    e->origin = origin;
    if (int rc = e->upload(problem, 1)) return rc;
    if (int rc = e->solve(params, nullptr, solution, trace)) return rc;
    std::vector<ChunkRecord> recs(1, record_of(e));
    fold(recs);
    res_begin.assign({0, 1});
    resident_B = 1;
    return PSULVSB_OK;
  }

  int solve_sharded(Comm* comm, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                    psulvsb_solution_t* solution, psulvsb_trace_t* trace) {
    Engine* e = eng[0];
    e->comm = comm;
    const int rc = solve_one(params, problem, solution, trace);
    e->comm = nullptr;
    return rc;
  }

  // evenly sized chunks of at most chunk_size() registrations
  static void partition(int B, int parts, std::vector<int>& begin) {
    begin.resize((size_t)parts + 1);
    for (int c = 0; c <= parts; ++c) begin[(size_t)c] = (int)((long long)B * c / parts);
  }

  int run_parallel(int n_workers, const std::function<int(int)>& work) {
    std::vector<int> rcs((size_t)n_workers, PSULVSB_OK);
    std::vector<std::string> msgs((size_t)n_workers);
    auto body = [&](int w) {
      const int rc = work(w);
      rcs[(size_t)w] = rc;
      if (rc) msgs[(size_t)w] = psulvsb_last_error();  // (the message is thread-local: carry it to the caller)
    };
    std::vector<std::thread> th;
    for (int w = 1; w < n_workers; ++w) th.emplace_back(body, w);
    body(0);
    for (auto& t : th) t.join();
    for (int w = 0; w < n_workers; ++w)
      if (rcs[(size_t)w]) return fail(rcs[(size_t)w], msgs[(size_t)w]);
    return PSULVSB_OK;
  }

  int solve_batch(const psulvsb_params_t* params, const psulvsb_problem_t* problems, int B, const uint64_t* seeds,
                  psulvsb_solution_t* solutions) {
    if (!params) return fail(PSULVSB_ERR_INVALID, "solve_batch: null params");
    drain();
    resident_B = 0;
    PSU_CUDA(cudaSetDevice(device));
    const int ch = chunk_size();
    const int n_chunks = (B + ch - 1) / ch;
    if (n_chunks > lane_count()) {
      // more chunks than lanes: through the queue of the pipelined calls, whose extra worker uploads the next chunk
      // while the lanes solve (only the first chunk's upload is exposed)
      uint64_t ticket = 0;
      if (int rc = submit(params, problems, B, seeds, solutions, &ticket)) return rc;
      return wait(ticket);
    }
    const int n_workers = n_chunks < lane_count() ? n_chunks : lane_count();
    if (int rc = ensure_engines(n_workers)) return rc;
    std::vector<int> begin;
    partition(B, n_chunks, begin);
    std::vector<uint64_t> own_seeds;
    if (!seeds && n_chunks > 1) {  // the default seed of a problem follows its index in the CALLER's batch
      own_seeds.resize((size_t)B);
      for (int b = 0; b < B; ++b) own_seeds[(size_t)b] = params->seed + (uint64_t)b;
      seeds = own_seeds.data();
    }
    PSU_CUDA(cudaEventRecord(origin, eng[0]->st));
    std::vector<ChunkRecord> recs((size_t)n_chunks);
    std::atomic<int> next(0);
    const int rc = run_parallel(n_workers, [&](int w) -> int {
      Engine* e = eng[(size_t)w];
      e->origin = origin;
      for (int c = next.fetch_add(1); c < n_chunks; c = next.fetch_add(1)) {
        const int b0 = begin[(size_t)c], nb = begin[(size_t)c + 1] - b0;
        {
          std::lock_guard<std::mutex> up(upload_mu);  // (see worker_main)
          if (int r = e->upload(problems + b0, nb)) return r;
        }
        if (int r = e->solve(params, seeds ? seeds + b0 : nullptr, solutions + b0, nullptr)) return r;
        recs[(size_t)c] = record_of(e);
      }
      return PSULVSB_OK;
    });
    if (rc) return rc;
    fold(recs);
    if (n_chunks == 1) {  // the batch is still resident on the first engine
      res_begin.assign({0, B});
      resident_B = B;
    }
    return PSULVSB_OK;
  }

  int upload(const psulvsb_problem_t* problems, int B) {
    drain();
    resident_B = 0;
    PSU_CUDA(cudaSetDevice(device));
    const int ch = chunk_size();
    int parts = (B + ch - 1) / ch;
    if (parts > lane_count()) parts = lane_count();  // resident chunks all run at once: one engine each
    if (int rc = ensure_engines(parts)) return rc;
    partition(B, parts, res_begin);
    for (int e = 0; e < parts; ++e)
      if (int rc = eng[(size_t)e]->upload(problems + res_begin[(size_t)e], res_begin[(size_t)e + 1] - res_begin[(size_t)e]))
        return rc;
    resident_B = B;
    return PSULVSB_OK;
  }

  // Every array of the batch must be device (or managed) memory of this handle's device: a kernel reading a host
  // address would fault the device, so anything else is refused before any device work.
  int check_device_pointers(const psulvsb_problem_t* problems, int B) {
    for (int b = 0; b < B; ++b) {
      const psulvsb_problem_t& p = problems[b];
      const void* arr[6] = {p.src, p.dst, p.ori_src, p.ori_dst, p.keep_mask, p.reduce_map};
      static const char* const names[6] = {"src", "dst", "ori_src", "ori_dst", "keep_mask", "reduce_map"};
      for (int k = 0; k < 6; ++k) {
        cudaPointerAttributes a;
        const cudaError_t e = cudaPointerGetAttributes(&a, arr[k]);
        if (e != cudaSuccess) cudaGetLastError();
        const bool ok = e == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) &&
                        a.device == device;
        if (!ok)
          return fail(PSULVSB_ERR_INVALID, "upload_device: problem " + std::to_string(b) + ": " + names[k] +
                                               " is not device memory of device " + std::to_string(device));
      }
    }
    return PSULVSB_OK;
  }

  // psulvsb_batch_upload_device: the split of upload, each engine's copy ordered after the caller's stream
  int upload_device(cudaStream_t caller, const psulvsb_problem_t* problems, int B) {
    drain();
    resident_B = 0;
    for (int b = 0; b < B; ++b)
      if (int rc = check_problem(problems[b], b)) return rc;
    PSU_CUDA(cudaSetDevice(device));
    if (int rc = check_device_pointers(problems, B)) return rc;
    const int ch = chunk_size();
    int parts = (B + ch - 1) / ch;
    if (parts > lane_count()) parts = lane_count();
    if (int rc = ensure_engines(parts)) return rc;
    partition(B, parts, res_begin);
    if (!ready) PSU_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    PSU_CUDA(cudaEventRecord(ready, caller));
    int rc = PSULVSB_OK;
    for (int e = 0; e < parts && !rc; ++e)
      rc = eng[(size_t)e]->upload_device_begin(problems + res_begin[(size_t)e],
                                               res_begin[(size_t)e + 1] - res_begin[(size_t)e], ready);
    if (rc) {
      // (the caller's buffers are not read after the call returns, whatever it returns)
      for (int e = 0; e < parts; ++e) cudaStreamSynchronize(eng[(size_t)e]->st);
      return rc;
    }
    for (int e = 0; e < parts; ++e)
      if (int r = eng[(size_t)e]->upload_device_finish(res_begin[(size_t)e])) {
        for (int f = e + 1; f < parts; ++f) cudaStreamSynchronize(eng[(size_t)f]->st);
        return r;
      }
    resident_B = B;
    return PSULVSB_OK;
  }

  int solve_resident(const psulvsb_params_t* params, const uint64_t* seeds, psulvsb_solution_t* solutions,
                     psulvsb_trace_t* trace_first) {
    drain();
    if (resident_B <= 0) return fail(PSULVSB_ERR_INVALID, "solve: nothing uploaded");
    if (!params) return fail(PSULVSB_ERR_INVALID, "solve: null params");
    PSU_CUDA(cudaSetDevice(device));
    const int parts = (int)res_begin.size() - 1;
    std::vector<uint64_t> own_seeds;
    if (!seeds && parts > 1) {
      own_seeds.resize((size_t)resident_B);
      for (int b = 0; b < resident_B; ++b) own_seeds[(size_t)b] = params->seed + (uint64_t)b;
      seeds = own_seeds.data();
    }
    for (int e = 0; e < parts; ++e) PSU_CUDA(cudaStreamSynchronize(eng[(size_t)e]->st));  // pending input copies
    PSU_CUDA(cudaEventRecord(origin, eng[0]->st));
    std::vector<ChunkRecord> recs((size_t)parts);
    const int rc = run_parallel(parts, [&](int w) -> int {
      Engine* e = eng[(size_t)w];
      e->origin = origin;
      const int b0 = res_begin[(size_t)w];
      if (int r = e->solve(params, seeds ? seeds + b0 : nullptr, solutions + b0, w == 0 ? trace_first : nullptr)) return r;
      recs[(size_t)w] = record_of(e);
      return PSULVSB_OK;
    });
    if (rc) {
      // a failed solve leaves the engines' resident inputs intact; nothing to undo
      return rc;
    }
    fold(recs);
    return PSULVSB_OK;
  }
};

// ---- C-linkage-free façade used by capi.cu ---------------------------------------------------
int pool_create(EnginePool** out, int device) {
  EnginePool* p = new EnginePool();
  const int rc = p->init(device);
  if (rc) {
    delete p;
    *out = nullptr;
    return rc;
  }
  *out = p;
  return PSULVSB_OK;
}
void pool_destroy(EnginePool* p) { delete p; }
int pool_set_batching(EnginePool* p, int chunk, int lanes) {
  if (chunk < 0 || lanes < 0 || lanes > 16) return fail(PSULVSB_ERR_INVALID, "set_batching: chunk >= 0, 0 <= lanes <= 16");
  p->drain();
  p->stop_workers();  // (the worker threads follow the lane count; they restart with the next submit)
  p->chunk = chunk;
  p->lanes = lanes;
  p->resident_B = 0;  // the resident partition followed the old setting
  return p->ensure_engines((int)p->eng.size());
}
int pool_set_host_threads(EnginePool* p, int n) {
  if (n < 0) return fail(PSULVSB_ERR_INVALID, "set_host_threads: n >= 0");
  p->host_threads = n;
  return p->ensure_engines((int)p->eng.size());
}
int pool_solve_one(EnginePool* p, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                   psulvsb_solution_t* solution, psulvsb_trace_t* trace) {
  return p->solve_one(params, problem, solution, trace);
}
int pool_solve_batch(EnginePool* p, const psulvsb_params_t* params, const psulvsb_problem_t* problems, int B,
                     const uint64_t* seeds, psulvsb_solution_t* solutions) {
  return p->solve_batch(params, problems, B, seeds, solutions);
}
int pool_submit(EnginePool* p, const psulvsb_params_t* params, const psulvsb_problem_t* problems, int B,
                const uint64_t* seeds, psulvsb_solution_t* solutions, uint64_t* ticket) {
  return p->submit(params, problems, B, seeds, solutions, ticket);
}
int pool_wait(EnginePool* p, uint64_t ticket) { return p->wait(ticket); }
int pool_solve_sharded(EnginePool* p, Comm* comm, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                       psulvsb_solution_t* solution, psulvsb_trace_t* trace) {
  return p->solve_sharded(comm, params, problem, solution, trace);
}
int pool_upload(EnginePool* p, const psulvsb_problem_t* problems, int B) { return p->upload(problems, B); }
int pool_upload_device(EnginePool* p, void* stream, const psulvsb_problem_t* problems, int B) {
  return p->upload_device(static_cast<cudaStream_t>(stream), problems, B);
}
int pool_solve_resident(EnginePool* p, const psulvsb_params_t* params, const uint64_t* seeds,
                        psulvsb_solution_t* solutions, psulvsb_trace_t* trace_first) {
  return p->solve_resident(params, seeds, solutions, trace_first);
}
int pool_batch_size(const EnginePool* p) { return p->resident_B; }
long long pool_launch_count(const EnginePool* p) { return p->launch_count(); }
double pool_last_device_ms(const EnginePool* p) { return p->last_ms; }
double pool_last_stage_ms(const EnginePool* p, int which) { return (which >= 0 && which < 5) ? p->stage_ms[which] : 0.0; }
int pool_last_ticks(const EnginePool* p) { return p->last_ticks; }
int pool_last_chunk_ticks(const EnginePool* p, int* out, int cap) {
  const int n = (int)p->chunk_ticks.size();
  for (int i = 0; i < n && i < cap; ++i) out[i] = p->chunk_ticks[(size_t)i];
  return n;
}

}  // namespace psulvsb
