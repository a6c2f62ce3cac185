// capi.cu -- the C ABI of libpsulvsb_b200.so (include/psulvsb.h): argument checking, error plumbing,
// single-job descriptors for the stage entry points, and the handle API over the batch engine.
// Nothing throws across this boundary and there is no CPU fallback.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "common.cuh"
#include "engine.cuh"

namespace psulvsb {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

int sm_count() {
  static int cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

DebugKnobs& debug_knobs() {
  static DebugKnobs k;
  return k;
}

int need_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return fail(PSULVSB_ERR_NO_DEVICE, "no CUDA device available (there is no CPU fallback)");
  }
  return PSULVSB_OK;
}

namespace {

// single job descriptor -> device, freed in stream order after the kernels that read it
template <typename T>
struct DeviceJob {
  T* d = nullptr;
  cudaStream_t st;
  explicit DeviceJob(cudaStream_t s) : st(s) {}
  int put(const T& h) {
    PSU_CUDA(cudaMallocAsync((void**)&d, sizeof(T), st));
    PSU_CUDA(cudaMemcpyAsync(d, &h, sizeof(T), cudaMemcpyHostToDevice, st));
    return PSULVSB_OK;
  }
  ~DeviceJob() {
    if (d) cudaFreeAsync(d, st);
  }
};

}  // namespace
}  // namespace psulvsb

using namespace psulvsb;

struct psulvsb_handle_s {
  EnginePool* pool;
  Comm* comm;
  int device;
};

extern "C" {

int psulvsb_version(void) { return PSULVSB_VERSION; }

const char* psulvsb_last_error(void) { return g_last_error.c_str(); }

void psulvsb_default_params(psulvsb_params_t* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  p->noise_bound = 0.01;             // registration.h:383
  p->cbar2 = 1;                      // registration.h:388
  p->estimate_scaling = 1;           // registration.h:396
  p->rotation_max_iterations = 100;  // registration.h:416
  p->rotation_gnc_factor = 1.4;      // registration.h:411
  p->rotation_cost_threshold = 1e-6; // registration.h:426
  p->inlier_selection_mode = 0;      // PMC_EXACT, registration.h:443
  p->kcore_heuristic_threshold = 0.5;
  p->score_noise_bound = 0.01;       // registration.cc:33
  p->inloop_noise_bound = 0.05;      // registration.cc:938
  p->inloop_cbar2 = 1;               // registration.cc:939
  p->inloop_max_iterations = 100;    // registration.cc:941
  p->inloop_gnc_factor = 1.4;        // registration.cc:942
  p->inloop_cost_threshold = 0.005;  // registration.cc:945
  p->rotation_similar = 0.01;        // registration.cc:48
  p->local_max_iter = 10;            // registration.cc:49
  p->tpro_host = 0.99;               // registration.cc:772
  p->tpro_local = 0.99;              // registration.cc:898
  p->host_round_limit = 5;           // registration.cc:781
  p->wallclock_cap_s = 60.0;         // registration.cc:1475
  p->self_update = 1;                // registration.cc:786-832
  p->seed = 0;
}

int psulvsb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int psulvsb_create(psulvsb_handle_t* out, int device) {
  if (!out) return fail(PSULVSB_ERR_INVALID, "psulvsb_create: out is NULL");
  *out = nullptr;
  if (int rc = need_device()) return rc;
  psulvsb_handle_s* h = new (std::nothrow) psulvsb_handle_s();
  if (!h) return fail(PSULVSB_ERR_INTERNAL, "out of host memory");
  h->comm = nullptr;
  h->device = device;
  const int rc = pool_create(&h->pool, device);
  if (rc) {
    delete h;
    return rc;
  }
  *out = h;
  return PSULVSB_OK;
}

int psulvsb_destroy(psulvsb_handle_t h) {
  if (!h) return PSULVSB_OK;
  comm_destroy(h->comm);
  pool_destroy(h->pool);
  delete h;
  return PSULVSB_OK;
}

int psulvsb_solve(psulvsb_handle_t h, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                  psulvsb_solution_t* solution, psulvsb_trace_t* trace) {
  if (!h || !params || !problem || !solution) return fail(PSULVSB_ERR_INVALID, "psulvsb_solve: NULL argument");
  return pool_solve_one(h->pool, params, problem, solution, trace);
}

int psulvsb_solve_batch(psulvsb_handle_t h, const psulvsb_params_t* params, const psulvsb_problem_t* problems, int B,
                        const uint64_t* seeds, psulvsb_solution_t* solutions) {
  if (!h || !params || !problems || !solutions || B <= 0)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_solve_batch: NULL argument or B <= 0");
  return pool_solve_batch(h->pool, params, problems, B, seeds, solutions);
}

int psulvsb_batch_submit(psulvsb_handle_t h, const psulvsb_params_t* params, const psulvsb_problem_t* problems, int B,
                         const uint64_t* seeds, psulvsb_solution_t* solutions, uint64_t* ticket) {
  if (!h || !params || !problems || !solutions || !ticket || B <= 0)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_batch_submit: NULL argument or B <= 0");
  return pool_submit(h->pool, params, problems, B, seeds, solutions, ticket);
}

int psulvsb_batch_wait(psulvsb_handle_t h, uint64_t ticket) {
  if (!h) return fail(PSULVSB_ERR_INVALID, "psulvsb_batch_wait: NULL handle");
  return pool_wait(h->pool, ticket);
}

int psulvsb_batch_upload(psulvsb_handle_t h, const psulvsb_problem_t* problems, int B) {
  if (!h || !problems || B <= 0) return fail(PSULVSB_ERR_INVALID, "psulvsb_batch_upload: NULL argument or B <= 0");
  return pool_upload(h->pool, problems, B);
}

int psulvsb_batch_upload_device(psulvsb_handle_t h, void* stream, const psulvsb_problem_t* problems, int B) {
  if (int rc = need_device()) return rc;
  if (!h || !problems || B <= 0)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_batch_upload_device: NULL argument or B <= 0");
  return pool_upload_device(h->pool, stream, problems, B);
}

int psulvsb_batch_solve_resident(psulvsb_handle_t h, const psulvsb_params_t* params, const uint64_t* seeds,
                                 psulvsb_solution_t* solutions, int n_solutions) {
  if (!h || !params || !solutions) return fail(PSULVSB_ERR_INVALID, "psulvsb_batch_solve_resident: NULL argument");
  const int B = pool_batch_size(h->pool);
  if (B <= 0) return fail(PSULVSB_ERR_INVALID, "psulvsb_batch_solve_resident: nothing is resident (upload first)");
  if (n_solutions != B)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_batch_solve_resident: " + std::to_string(n_solutions) +
                                         " solution slots for a resident batch of " + std::to_string(B));
  return pool_solve_resident(h->pool, params, seeds, solutions, nullptr);
}

int psulvsb_debug_set(const char* name, double value) {
  if (!name) return fail(PSULVSB_ERR_INVALID, "psulvsb_debug_set: NULL name");
  DebugKnobs& k = debug_knobs();
  const std::string n(name);
  if (n == "gnc_deep_margin") k.gnc_deep_margin = value;
  else if (n == "sample_list_cap_test") k.sample_list_cap_test = (int)value;
  else if (n == "k1_variant") {
    if (value != 0 && value != 1 && value != 2 && value != 4)
      return fail(PSULVSB_ERR_INVALID, "psulvsb_debug_set: k1_variant must be 0 (automatic), 1, 2 or 4");
    k.k1_variant = (int)value;
  } else if (n == "edge_wide") k.edge_wide = (int)value;
  else if (n == "reset") k = DebugKnobs();
  else return fail(PSULVSB_ERR_INVALID, "psulvsb_debug_set: unknown switch " + n);
  return PSULVSB_OK;
}

int psulvsb_batch_resident_size(psulvsb_handle_t h) { return h ? pool_batch_size(h->pool) : 0; }

int psulvsb_set_batching(psulvsb_handle_t h, int chunk, int lanes) {
  if (!h) return fail(PSULVSB_ERR_INVALID, "psulvsb_set_batching: NULL handle");
  return pool_set_batching(h->pool, chunk, lanes);
}

int psulvsb_set_host_threads(psulvsb_handle_t h, int n) {
  if (!h) return fail(PSULVSB_ERR_INVALID, "psulvsb_set_host_threads: NULL handle");
  return pool_set_host_threads(h->pool, n);
}

long long psulvsb_launch_count(psulvsb_handle_t h) { return h ? pool_launch_count(h->pool) : 0; }
double psulvsb_last_device_ms(psulvsb_handle_t h) { return h ? pool_last_device_ms(h->pool) : 0.0; }
double psulvsb_last_stage_ms(psulvsb_handle_t h, int which) { return h ? pool_last_stage_ms(h->pool, which) : 0.0; }
int psulvsb_last_ticks(psulvsb_handle_t h) { return h ? pool_last_ticks(h->pool) : 0; }
int psulvsb_last_chunk_ticks(psulvsb_handle_t h, int* out, int cap) {
  if (!h || (cap > 0 && !out)) return 0;
  return pool_last_chunk_ticks(h->pool, out, cap);
}

/* ---------------------------------------------------------------------------------------------- */
/* stage entry points                                                                              */
/* ---------------------------------------------------------------------------------------------- */

int psulvsb_pack_points(void* stream, const double* d_pts, int n, const double center[3], void* d_out_float4) {
  if (int rc = need_device()) return rc;
  if (!d_pts || !d_out_float4 || n < 0) return fail(PSULVSB_ERR_INVALID, "psulvsb_pack_points: bad argument");
  return launch_pack_points((cudaStream_t)stream, d_pts, n, center, (float4*)d_out_float4);
}

int psulvsb_consistency_mask_rows(void* stream, const void* d_src_f4, const void* d_dst_f4, const double* d_src64,
                                  const double* d_dst64, int n, int row_begin, int row_end, double beta,
                                  double coord_bound, uint32_t* d_mask, int row_stride_words, uint32_t* d_row_counts,
                                  unsigned long long* d_border_count) {
  if (int rc = need_device()) return rc;
  if (!d_src_f4 || !d_dst_f4 || !d_src64 || !d_dst64 || !d_mask)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_consistency_mask: NULL array");
  if (n < 1 || row_begin < 0 || row_end > n || row_begin > row_end)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_consistency_mask: bad n / row range");
  if (row_stride_words < (n + 31) / 32)
    return fail(PSULVSB_ERR_CAPACITY, "psulvsb_consistency_mask: row_stride_words < ceil(n / 32)");
  if (!(beta >= 0.0) || !(coord_bound >= 0.0) || !std::isfinite(beta) || !std::isfinite(coord_bound))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_consistency_mask: beta / coord_bound must be finite and >= 0");
  if (((uintptr_t)d_src_f4 & 15) || ((uintptr_t)d_dst_f4 & 15))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_consistency_mask: float4 arrays must be 16-byte aligned");
  if (row_begin == row_end) return PSULVSB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // the kernel streams pair-interleaved records (common.cuh il_store): built here from the caller's per-point ones
  float4* il = nullptr;
  const size_t nrec = il_records((size_t)n);
  PSU_CUDA(cudaMallocAsync((void**)&il, sizeof(float4) * 2 * nrec, st));
  struct IlFree {
    float4* p;
    cudaStream_t s;
    ~IlFree() { cudaFreeAsync(p, s); }
  } il_free{il, st};
  if (int rc = launch_interleave_points(st, (const float4*)d_src_f4, n, il)) return rc;
  if (int rc = launch_interleave_points(st, (const float4*)d_dst_f4, n, il + nrec)) return rc;
  K1Job j;
  std::memset(&j, 0, sizeof(j));
  j.src = il;
  j.dst = il + nrec;
  j.src64 = d_src64;
  j.dst64 = d_dst64;
  j.n = n;
  j.row_begin = row_begin;
  j.row_end = row_end;
  j.c = make_k1_consts(beta, coord_bound);
  j.mask = d_mask;
  j.stride = row_stride_words;
  j.row_counts = d_row_counts;
  j.border = d_border_count;
  j.active = 1;
  if (d_row_counts) PSU_CUDA(cudaMemsetAsync(d_row_counts + row_begin, 0, sizeof(uint32_t) * (size_t)(row_end - row_begin), st));
  // the kernel writes only the words at or right of each row's diagonal tile: define the rest as zeros
  PSU_CUDA(cudaMemsetAsync(d_mask + (size_t)row_begin * row_stride_words, 0,
                           sizeof(uint32_t) * (size_t)(row_end - row_begin) * row_stride_words, st));
  DeviceJob<K1Job> dj(st);
  if (int rc = dj.put(j)) return rc;
  return launch_consistency_mask(st, dj.d, 1, n, row_end - row_begin, (row_stride_words & 7) == 0);
}

int psulvsb_consistency_mask(void* stream, const void* d_src_f4, const void* d_dst_f4, const double* d_src64,
                             const double* d_dst64, int n, double beta, double coord_bound, uint32_t* d_mask,
                             int row_stride_words, uint32_t* d_row_counts, unsigned long long* d_border_count) {
  return psulvsb_consistency_mask_rows(stream, d_src_f4, d_dst_f4, d_src64, d_dst64, n, 0, n, beta, coord_bound, d_mask,
                                       row_stride_words, d_row_counts, d_border_count);
}

int psulvsb_mask_symmetrize(void* stream, uint32_t* d_mask, int n, int row_stride_words) {
  if (int rc = need_device()) return rc;
  if (!d_mask || n < 1 || row_stride_words < (n + 31) / 32)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_mask_symmetrize: bad argument");
  return launch_symmetrize((cudaStream_t)stream, d_mask, n, row_stride_words);
}

int psulvsb_compact_edges(void* stream, const uint32_t* d_mask, int n, int row_stride_words,
                          const uint32_t* d_row_counts, unsigned long long* d_row_offsets, void* d_edges_uint2,
                          unsigned long long edge_capacity, unsigned long long* d_n_edges) {
  if (int rc = need_device()) return rc;
  if (!d_mask || !d_row_counts || !d_row_offsets || n < 1 || row_stride_words < (n + 31) / 32)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_compact_edges: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  CompactJob j;
  std::memset(&j, 0, sizeof(j));
  j.mask = d_mask;
  j.n = n;
  j.stride = row_stride_words;
  j.row_counts = d_row_counts;
  j.offsets = d_row_offsets;
  j.edges = d_edges_uint2;
  j.cap = edge_capacity;
  j.n_edges = d_n_edges;
  j.active = 1;
  DeviceJob<CompactJob> dj(st);
  if (int rc = dj.put(j)) return rc;
  return launch_compact_edges(st, dj.d, 1, n, true, d_edges_uint2 != nullptr, false);
}

int psulvsb_ratio_reduced_set(void* stream, const double* d_src64, const double* d_dst64, int n, uint32_t* d_pair_bin,
                              void* d_edges_uint2, unsigned long long edge_capacity, unsigned long long* n_edges,
                              double* max_scale, unsigned int peak[2]) {
  if (!d_src64 || !d_dst64 || !n_edges || n < 2)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_ratio_reduced_set: NULL array / n_edges, or n < 2");
  if (int rc = need_device()) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t L = (size_t)n * (size_t)(n - 1) / 2;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = (off + 15) & ~(size_t)15;
    off = o + bytes;
    return o;
  };
  const size_t o_bins = d_pair_bin ? 0 : take(sizeof(uint32_t) * L);
  const size_t o_rmax = take(sizeof(double) * (size_t)n), o_bpi = take(sizeof(unsigned long long) * RATIO_MAX_GROWTHS),
               o_bps = take(sizeof(double) * RATIO_MAX_GROWTHS), o_bpn = take(sizeof(unsigned int)),
               o_fs = take(sizeof(double)), o_bad = take(sizeof(int)), o_peak = take(4 * sizeof(unsigned int)),
               o_cc = take(sizeof(unsigned int) * 3 * (size_t)n),
               o_co = take(sizeof(unsigned long long) * (3 * (size_t)n + 1)), o_ne = take(sizeof(unsigned long long));
  struct Scratch {
    char* p = nullptr;
    void* hist = nullptr;
    cudaStream_t s;
    ~Scratch() {
      if (p) cudaFreeAsync(p, s);
      if (hist) cudaFreeAsync(hist, s);
    }
  } scr;
  scr.s = st;
  PSU_CUDA(cudaMallocAsync((void**)&scr.p, off, st));
  std::vector<RatioJob> rj(1);
  RatioJob& j = rj[0];
  std::memset(&j, 0, sizeof(j));
  j.src64 = d_src64;
  j.dst64 = d_dst64;
  j.n = n;
  j.pair_bin = d_pair_bin ? d_pair_bin : reinterpret_cast<uint32_t*>(scr.p + o_bins);
  j.row_max = reinterpret_cast<double*>(scr.p + o_rmax);
  j.bp_idx = reinterpret_cast<unsigned long long*>(scr.p + o_bpi);
  j.bp_scale = reinterpret_cast<double*>(scr.p + o_bps);
  j.bp_n = reinterpret_cast<unsigned int*>(scr.p + o_bpn);
  j.final_scale = reinterpret_cast<double*>(scr.p + o_fs);
  j.bad = reinterpret_cast<int*>(scr.p + o_bad);
  j.peak = reinterpret_cast<unsigned int*>(scr.p + o_peak);
  j.class_counts = reinterpret_cast<unsigned int*>(scr.p + o_cc);
  j.class_offsets = reinterpret_cast<unsigned long long*>(scr.p + o_co);
  j.n_edges = reinterpret_cast<unsigned long long*>(scr.p + o_ne);
  j.active = 1;
  DeviceJob<RatioJob> dj(st);
  if (int rc = dj.put(j)) return rc;
  auto arena = [&](size_t bytes) -> void* {
    const cudaError_t e = cudaMallocAsync(&scr.hist, bytes, st);
    if (e == cudaSuccess) return scr.hist;
    scr.hist = nullptr;
    fail(PSULVSB_ERR_CUDA, std::string("psulvsb_ratio_reduced_set: histogram allocation: ") + cudaGetErrorString(e));
    return nullptr;
  };
  if (int rc = ratio_count(st, rj, dj.d, n, arena, nullptr, nullptr)) return rc;
  unsigned long long ne = 0;
  double fs = 0.0;
  unsigned int pk[2] = {0u, 0u};
  PSU_CUDA(cudaMemcpyAsync(&ne, j.n_edges, sizeof(ne), cudaMemcpyDeviceToHost, st));
  PSU_CUDA(cudaMemcpyAsync(&fs, j.final_scale, sizeof(fs), cudaMemcpyDeviceToHost, st));
  PSU_CUDA(cudaMemcpyAsync(pk, j.peak, sizeof(pk), cudaMemcpyDeviceToHost, st));
  PSU_CUDA(cudaStreamSynchronize(st));
  *n_edges = ne;
  if (max_scale) *max_scale = fs;
  if (peak) {
    peak[0] = pk[0];
    peak[1] = pk[1];
  }
  if (!d_edges_uint2) return PSULVSB_OK;
  if (ne > edge_capacity)
    return fail(PSULVSB_ERR_CAPACITY, "psulvsb_ratio_reduced_set: " + std::to_string(ne) + " edges, capacity " +
                                          std::to_string(edge_capacity));
  j.edges = d_edges_uint2;
  j.cap = edge_capacity;
  if (int rc = ratio_emit(st, rj, dj.d, n, false)) return rc;
  PSU_CUDA(cudaStreamSynchronize(st));
  return PSULVSB_OK;
}

unsigned long long psulvsb_sample_default_max_draws(unsigned long long n, unsigned long long count) {
  return sample_default_max_draws(n, count);
}

unsigned long long psulvsb_sample_workspace_bytes(unsigned long long n, unsigned long long count,
                                                  unsigned long long max_draws) {
  if (max_draws == 0) max_draws = sample_default_max_draws(n, count);
  return ((sample_table_words(n, max_draws) * sizeof(uint32_t) + 15) & ~15ull) +
         sample_chunk_slots(max_draws) * sizeof(unsigned long long) + 16 +
         sample_list_counters() * sizeof(unsigned int) + sample_list_entries(n, max_draws) * sizeof(uint32_t);
}

int psulvsb_sample(void* stream, uint64_t seed, uint32_t domain, uint32_t event, unsigned long long n,
                   unsigned long long count, unsigned long long max_draws, uint32_t* d_out, void* d_work,
                   unsigned long long* d_status) {
  if (int rc = need_device()) return rc;
  if (!d_out || !d_work || !d_status) return fail(PSULVSB_ERR_INVALID, "psulvsb_sample: NULL array");
  if (n == 0 || count > n) return fail(PSULVSB_ERR_INVALID, "psulvsb_sample: need 0 < n and count <= n");
  if (n >= 0x7FFFFFFFull) return fail(PSULVSB_ERR_UNSUPPORTED, "psulvsb_sample: n must fit the 31-bit draws");
  if (max_draws == 0) max_draws = sample_default_max_draws(n, count);
  if (max_draws >= 0xFFFFFFFFull) return fail(PSULVSB_ERR_UNSUPPORTED, "psulvsb_sample: max_draws must be < 2^32 - 1");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t first_bytes = (sample_table_words(n, max_draws) * sizeof(uint32_t) + 15) & ~15ull;
  const size_t slots = sample_chunk_slots(max_draws);
  PSU_CUDA(cudaMemsetAsync(d_work, 0, first_bytes, st));
  PSU_CUDA(cudaMemsetAsync((char*)d_work + first_bytes + slots * sizeof(unsigned long long), 0, 16, st));
  PSU_CUDA(cudaMemsetAsync(d_status, 0, sizeof(unsigned long long), st));
  if (count == 0) return PSULVSB_OK;
  SampleJob j;
  std::memset(&j, 0, sizeof(j));
  j.seed = seed;
  j.domain = domain;
  j.event = event;
  j.n = n;
  j.count = count;
  j.max_draws = max_draws;
  j.first = (uint32_t*)d_work;
  j.chunk_prefix = (unsigned long long*)((char*)d_work + first_bytes);
  j.ticket = (unsigned int*)((char*)d_work + first_bytes + slots * sizeof(unsigned long long));
  {
    // bucket-list scratch behind the ticket: counters (zeroed), then the lists
    char* p = (char*)d_work + first_bytes + slots * sizeof(unsigned long long) + 16;
    j.bcount = (unsigned int*)p;
    PSU_CUDA(cudaMemsetAsync(p, 0, sample_list_counters() * sizeof(unsigned int), st));
    j.blist_cap = sample_list_entries(n, max_draws);
    j.blist = j.blist_cap ? (uint32_t*)(p + sample_list_counters() * sizeof(unsigned int)) : nullptr;
  }
  j.out = d_out;
  j.status = d_status;
  j.active = 1;
  DeviceJob<SampleJob> dj(st);
  if (int rc = dj.put(j)) return rc;
  return launch_sample(st, dj.d, 1, max_draws, n);
}

int psulvsb_philox_fill(void* stream, uint64_t seed, uint32_t domain, uint32_t event, unsigned long long first_k,
                        unsigned long long count, uint32_t* d_out_rand31) {
  if (int rc = need_device()) return rc;
  if (!d_out_rand31 && count) return fail(PSULVSB_ERR_INVALID, "psulvsb_philox_fill: NULL output");
  return launch_philox_fill((cudaStream_t)stream, seed, domain, event, first_k, count, d_out_rand31);
}

int psulvsb_gnc_tls_rotation(void* stream, const double* d_src64, const double* d_dst64, const void* d_edges_uint2,
                             unsigned long long K, double inv_scale, double noise_bound, int max_iterations,
                             double gnc_factor, double cost_threshold, const double* d_R_init, double* d_weights,
                             double* d_R, uint8_t* d_inliers, int* d_info, double* d_cost) {
  if (int rc = need_device()) return rc;
  if (!d_src64 || !d_dst64 || (!d_edges_uint2 && K) || !d_R || (!d_weights && K))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_gnc_tls_rotation: NULL array");
  if (max_iterations < 0) return fail(PSULVSB_ERR_INVALID, "psulvsb_gnc_tls_rotation: max_iterations < 0");
  if (K >= 0x7FFFFFF0ull) return fail(PSULVSB_ERR_UNSUPPORTED, "psulvsb_gnc_tls_rotation: K must fit 31 bits");
  cudaStream_t st = (cudaStream_t)stream;
  GncJob j;
  std::memset(&j, 0, sizeof(j));
  j.src = d_src64;
  j.dst = d_dst64;
  j.edges = (const uint2*)d_edges_uint2;
  j.K = K;
  j.inv_scale = inv_scale;
  j.noise_bound = noise_bound;
  j.gnc_factor = gnc_factor;
  j.cost_threshold = cost_threshold;
  j.max_iterations = max_iterations;
  j.use_init = d_R_init ? 1 : 0;
  if (d_R_init) PSU_CUDA(cudaMemcpyAsync(j.R_init, d_R_init, sizeof(double) * 9, cudaMemcpyDeviceToHost, st));
  if (d_R_init) PSU_CUDA(cudaStreamSynchronize(st));
  j.weights = d_weights;
  j.lv = nullptr;
  j.lv_cap = 0;
  j.R_out = d_R;
  j.inliers = d_inliers;
  j.point_flags = nullptr;
  j.n_points = 0;
  j.info = d_info;
  j.cost = d_cost;
  j.active = 1;
  DeviceJob<GncJob> dj(st);
  if (int rc = dj.put(j)) return rc;
  int cap = (int)((K + 7) / 8) + 32;
  cap = (cap + 31) & ~31;
  return launch_gnc_tls(st, dj.d, 1, cap, 8);
}

int psulvsb_gnc_tls_rotation_batch(void* stream, const double* d_src64, const double* d_dst64, int n_points,
                                   const void* d_edges_uint2, unsigned long long K, int n_jobs, double noise_bound,
                                   int max_iterations, double gnc_factor, double cost_threshold, int cluster,
                                   double* d_weights, double* d_lv, unsigned long long lv_cap, uint32_t* d_perm,
                                   double* d_R, uint8_t* d_inliers, int* d_info, long long* d_prof) {
  if (int rc = need_device()) return rc;
  if (!d_src64 || !d_dst64 || !d_edges_uint2 || !d_R || !d_weights || n_jobs < 1 || K < 1)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_gnc_tls_rotation_batch: bad argument");
  if (K >= 0x7FFFFFF0ull) return fail(PSULVSB_ERR_UNSUPPORTED, "psulvsb_gnc_tls_rotation_batch: K must fit 31 bits");
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<GncJob> jobs((size_t)n_jobs);
  for (int b = 0; b < n_jobs; ++b) {
    GncJob& j = jobs[(size_t)b];
    std::memset(&j, 0, sizeof(j));
    j.src = d_src64;
    j.dst = d_dst64;
    j.edges = (const uint2*)d_edges_uint2 + (size_t)b * K;
    j.K = K;
    j.inv_scale = 1.0;
    j.noise_bound = noise_bound;
    j.gnc_factor = gnc_factor;
    j.cost_threshold = cost_threshold;
    j.max_iterations = max_iterations;
    j.weights = d_weights + (size_t)b * K;
    j.lv = d_lv ? d_lv + (size_t)b * 6 * lv_cap : nullptr;
    j.lv_cap = d_lv ? lv_cap : 0;
    j.perm = (d_lv && d_perm) ? d_perm + (size_t)b * 2 * lv_cap : nullptr;
    j.R_out = d_R + (size_t)b * 9;
    j.inliers = d_inliers ? d_inliers + (size_t)b * K : nullptr;
    j.n_points = n_points;
    j.info = d_info ? d_info + (size_t)b * 4 : nullptr;
    j.prof = d_prof ? d_prof + (size_t)b * 8 : nullptr;
    j.active = 1;
  }
  struct AsyncJobs {  // freed on every exit path (stream-ordered, after the launch that reads it)
    GncJob* d = nullptr;
    double* red = nullptr;  // grid mode: the CTAs' partial results and arrival counters
    unsigned int* bar = nullptr;
    cudaStream_t st;
    explicit AsyncJobs(cudaStream_t s) : st(s) {}
    ~AsyncJobs() {
      if (d) cudaFreeAsync(d, st);
      if (red) cudaFreeAsync(red, st);
      if (bar) cudaFreeAsync(bar, st);
    }
  } dj(st);
  const bool grid_mode = cluster > 8;  // `cluster` CTAs per registration, launched cooperatively
  if (grid_mode) {
    PSU_CUDA(cudaMallocAsync((void**)&dj.red, sizeof(double) * (size_t)n_jobs * cluster * GNC_GRID_RED_DOUBLES, st));
    PSU_CUDA(cudaMallocAsync((void**)&dj.bar, sizeof(unsigned int) * (size_t)n_jobs, st));
    for (int b = 0; b < n_jobs; ++b) {
      jobs[(size_t)b].grid_red = dj.red + (size_t)b * cluster * GNC_GRID_RED_DOUBLES;
      jobs[(size_t)b].grid_bar = dj.bar + b;
    }
  }
  PSU_CUDA(cudaMallocAsync((void**)&dj.d, sizeof(GncJob) * (size_t)n_jobs, st));
  PSU_CUDA(cudaMemcpyAsync(dj.d, jobs.data(), sizeof(GncJob) * (size_t)n_jobs, cudaMemcpyHostToDevice, st));
  PSU_CUDA(cudaStreamSynchronize(st));  // jobs is pageable host memory
  if (!grid_mode && cluster != 1 && cluster != 2 && cluster != 4 && cluster != 8) cluster = gnc_cluster_for(n_jobs);
  int cap = (int)((K + (unsigned long long)cluster - 1) / (unsigned long long)cluster) + 32;
  cap = (cap + 31) & ~31;
  return launch_gnc_tls(st, dj.d, n_jobs, cap, cluster, 0);
}

int psulvsb_kabsch_batch(void* stream, const double* d_src64, const double* d_dst64, const void* d_edges_uint2,
                         const uint32_t* d_sets, int k, unsigned long long n_hyp, double* d_R, double* d_t) {
  if (int rc = need_device()) return rc;
  if (!d_src64 || !d_dst64 || !d_edges_uint2 || !d_sets || !d_R)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_kabsch_batch: NULL array");
  return launch_kabsch_batch((cudaStream_t)stream, d_src64, d_dst64, (const uint2*)d_edges_uint2, d_sets, k, n_hyp, d_R,
                             d_t);
}

int psulvsb_tls_translation(void* stream, const double* d_src64, const double* d_dst64, const uint8_t* d_point_flags,
                            int n, double scale, const double* d_R, double noise, const double* d_last_best,
                            double* d_t_out, int* d_n_points) {
  if (int rc = need_device()) return rc;
  if (!d_src64 || !d_dst64 || !d_point_flags || !d_R || !d_t_out)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_tls_translation: NULL array");
  return launch_tls_translation((cudaStream_t)stream, d_src64, d_dst64, d_point_flags, n, scale, d_R, noise, d_last_best,
                                d_t_out, d_n_points);
}

int psulvsb_estimate_normals(void* stream, const double* d_pts, int n, int k, const double viewpoint[3],
                             double* d_normals) {
  if (int rc = need_device()) return rc;
  if (!d_pts || !d_normals || n < 0) return fail(PSULVSB_ERR_INVALID, "psulvsb_estimate_normals: bad argument");
  return launch_knn_normals((cudaStream_t)stream, d_pts, n, k, viewpoint, d_normals);
}

int psulvsb_estimate_normals_host(const double* pts, int n, int k, const double viewpoint[3], double* normals) {
  if (int rc = need_device()) return rc;
  if (!pts || !normals || n < 0) return fail(PSULVSB_ERR_INVALID, "psulvsb_estimate_normals_host: bad argument");
  if (n == 0) return PSULVSB_OK;
  double *d_p = nullptr, *d_n = nullptr;
  const size_t bytes = sizeof(double) * 3 * (size_t)n;
  PSU_CUDA(cudaMalloc((void**)&d_p, bytes));
  if (cudaMalloc((void**)&d_n, bytes) != cudaSuccess) {
    cudaFree(d_p);
    return fail(PSULVSB_ERR_CUDA, "psulvsb_estimate_normals_host: cudaMalloc failed");
  }
  int rc = PSULVSB_OK;
  if (cudaMemcpy(d_p, pts, bytes, cudaMemcpyHostToDevice) != cudaSuccess) rc = fail(PSULVSB_ERR_CUDA, "H2D copy failed");
  if (!rc) rc = launch_knn_normals(nullptr, d_p, n, k, viewpoint, d_n);
  if (!rc && cudaMemcpy(normals, d_n, bytes, cudaMemcpyDeviceToHost) != cudaSuccess)
    rc = fail(PSULVSB_ERR_CUDA, std::string("normals kernel / D2H copy failed: ") + cudaGetErrorString(cudaGetLastError()));
  cudaFree(d_p);
  cudaFree(d_n);
  return rc;
}

unsigned long long psulvsb_max_clique_scratch_words(int n_vertices) {
  return n_vertices < 1 ? 0ull : (unsigned long long)clique_scratch_words(n_vertices);
}

int psulvsb_max_clique(void* stream, const void* d_edges_uint2, unsigned long long n_edges, int n_vertices,
                       uint32_t* d_adj, uint8_t* d_flags, int* d_size, int exact) {
  if (int rc = need_device()) return rc;
  if ((!d_edges_uint2 && n_edges) || !d_adj || !d_flags || !d_size || n_vertices < 1)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_max_clique: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  CliqueJob j;
  std::memset(&j, 0, sizeof(j));
  j.edges = (const uint2*)d_edges_uint2;
  j.n_edges = n_edges;
  j.filter = 0;
  j.n_vertices = n_vertices;
  j.adj = d_adj;
  j.stride = (n_vertices + 31) / 32;
  j.flags = d_flags;
  j.size = d_size;
  j.proven = d_size + 1;
  j.active = 1;
  DeviceJob<CliqueJob> dj(st);
  if (int rc = dj.put(j)) return rc;
  return launch_max_clique(st, dj.d, 1, n_vertices, j.stride, n_edges, exact != 0);
}

int psulvsb_score_batch(void* stream, const void* d_src_f4, const void* d_dst_f4, const double* d_src64,
                        const double* d_dst64, int n, const double* d_hyp, unsigned long long n_hyp,
                        unsigned long long hyp_begin, double scale, double tau, double coord_bound,
                        const double center_src[3], const double center_dst[3], uint32_t* d_counts,
                        unsigned long long* d_best, unsigned long long* d_border_count) {
  if (int rc = need_device()) return rc;
  if (!d_src_f4 || !d_dst_f4 || !d_src64 || !d_dst64 || !d_hyp || !d_counts)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_score_batch: NULL array");
  if (((uintptr_t)d_src_f4 & 15) || ((uintptr_t)d_dst_f4 & 15))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_score_batch: float4 arrays must be 16-byte aligned");
  if (!(tau >= 0.0) || !std::isfinite(tau) || !std::isfinite(scale) || !(coord_bound >= 0.0))
    return fail(PSULVSB_ERR_INVALID, "psulvsb_score_batch: bad tau / scale / coord_bound");
  return launch_score_batch((cudaStream_t)stream, (const float4*)d_src_f4, (const float4*)d_dst_f4, d_src64, d_dst64, n,
                            d_hyp, n_hyp, hyp_begin, scale, tau, coord_bound, center_src, center_dst, d_counts, d_best,
                            d_border_count);
}

/* ---------------------------------------------------------------------------------------------- */
/* multi-GPU: one process per GPU, one NCCL communicator per handle                                */
/* ---------------------------------------------------------------------------------------------- */

int psulvsb_comm_unique_id(void* out_id) {
  if (!out_id) return fail(PSULVSB_ERR_INVALID, "psulvsb_comm_unique_id: NULL");
  return comm_unique_id(out_id);
}

int psulvsb_comm_create(psulvsb_handle_t h, int rank, int world, const void* id) {
  if (!h || !id) return fail(PSULVSB_ERR_INVALID, "psulvsb_comm_create: NULL argument");
  if (h->comm) {
    comm_destroy(h->comm);
    h->comm = nullptr;
  }
  return comm_create(&h->comm, h->device, rank, world, id);
}

int psulvsb_comm_destroy(psulvsb_handle_t h) {
  if (!h) return PSULVSB_OK;
  comm_destroy(h->comm);
  h->comm = nullptr;
  return PSULVSB_OK;
}

int psulvsb_shard_row_range(int n, int rank, int world, int* begin, int* end) {
  if (!begin || !end || n < 0 || world < 1 || rank < 0 || rank >= world)
    return fail(PSULVSB_ERR_INVALID, "psulvsb_shard_row_range: bad argument");
  triangular_row_range(n, rank, world, begin, end);
  return PSULVSB_OK;
}

int psulvsb_comm_rank(psulvsb_handle_t h) { return h ? comm_rank(h->comm) : 0; }
int psulvsb_comm_world(psulvsb_handle_t h) { return h ? comm_world(h->comm) : 1; }

int psulvsb_comm_allreduce_sum_u32(psulvsb_handle_t h, void* stream, uint32_t* d_inout, unsigned long long n) {
  if (!h || !d_inout) return fail(PSULVSB_ERR_INVALID, "psulvsb_comm_allreduce_sum_u32: NULL argument");
  return comm_allreduce_sum_u32(h->comm, (cudaStream_t)stream, d_inout, (size_t)n);
}

int psulvsb_comm_allreduce_max_u64(psulvsb_handle_t h, void* stream, unsigned long long* d_inout, unsigned long long n) {
  if (!h || !d_inout) return fail(PSULVSB_ERR_INVALID, "psulvsb_comm_allreduce_max_u64: NULL argument");
  return comm_allreduce_max_u64(h->comm, (cudaStream_t)stream, d_inout, (size_t)n);
}

int psulvsb_score_batch_sharded(psulvsb_handle_t h, void* stream, const void* d_src_f4, const void* d_dst_f4,
                                const double* d_src64, const double* d_dst64, int n, const double* d_hyp,
                                unsigned long long n_hyp, unsigned long long hyp_begin, double scale, double tau,
                                double coord_bound, const double center_src[3], const double center_dst[3],
                                uint32_t* d_counts, unsigned long long* d_best, unsigned long long* d_border_count) {
  if (!h || !d_best) return fail(PSULVSB_ERR_INVALID, "psulvsb_score_batch_sharded: NULL handle / d_best");
  if (int rc = psulvsb_score_batch(stream, d_src_f4, d_dst_f4, d_src64, d_dst64, n, d_hyp, n_hyp, hyp_begin, scale, tau,
                                   coord_bound, center_src, center_dst, d_counts, d_best, d_border_count))
    return rc;
  // the global best = max of the packed keys (count << 32 | ~id): 8 bytes over NVLink, in-stream
  return comm_allreduce_max_u64(h->comm, (cudaStream_t)stream, d_best, 1);
}

int psulvsb_solve_sharded(psulvsb_handle_t h, const psulvsb_params_t* params, const psulvsb_problem_t* problem,
                          psulvsb_solution_t* solution, psulvsb_trace_t* trace) {
  if (!h || !params || !problem || !solution) return fail(PSULVSB_ERR_INVALID, "psulvsb_solve_sharded: NULL argument");
  return pool_solve_sharded(h->pool, h->comm, params, problem, solution, trace);
}

int psulvsb_score_one(void* stream, const double* d_src64, const double* d_dst64, int n, double scale,
                      const double* d_R, const double* d_t, double tau, uint8_t* d_inliers, double* d_residuals,
                      int* d_count) {
  if (int rc = need_device()) return rc;
  if (!d_src64 || !d_dst64 || !d_R || !d_t) return fail(PSULVSB_ERR_INVALID, "psulvsb_score_one: NULL array");
  cudaStream_t st = (cudaStream_t)stream;
  if (d_count) PSU_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int), st));
  return launch_score_one(st, d_src64, d_dst64, n, scale, d_R, d_t, tau, d_inliers, d_residuals, d_count);
}

}  // extern "C"
